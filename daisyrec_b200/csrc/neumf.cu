// neumf.cu -- NeuMF + BPR on the B200 path (SURVEY 8(a) row a14), fp32 tower on CUDA cores.
//
// Stands behind daisy/model/NeuMFRecommender.py (model_name == 'NeuMF'):
//   forward   :118-137  GMF = UG[u]*IG[i];  x0 = cat(UM[u], IM[i]);  L x (Dropout -> Linear -> ReLU);  Linear(2F, 1)
//   calc_loss :139-169  BPR + the regulariser as written, quirk included (:158,:160 use the GMF table for the MLP-neg term)
//   backward + optimizer.step (AbstractRecommender.py:125-126; dense Adam by default, NeuMFRecommender.py:74)
//   rank / full_rank / predict :171-232 (scores through the whole tower)
//
// One training step on a batch of B triples (R = 2B rows: pos rows [0,B), neg rows [B,2B)):
//   gather      A_0[R, 2D]  = cat(UM[u], IM[item])                      (lane group per row, 128-bit loads)
//   tower fwd   A_l = relu(A_{l-1} W_l^T + b_l)                         (tiled fp32 GEMM, fused bias + ReLU)
//   head        pred, BPR coefficient, loss + regulariser norms, GMF gradients (RED.ADD.F32x4), dZ_L, row counters
//   tower bwd   gW_l += (A_{l-1}^T dZ_l)^T (split-K, transposed atomic accumulate);  dZ_{l-1} = (dZ_l W_l) * [A_{l-1} > 0]
//   scatter     gUM[u] += dA_0[:, :D] (pos + neg rows), gIM[item] += dA_0[:, D:]
//   apply       the MF dense sweep (mf_bpr.cu) on the table pairs (UG,IG) and (UM,IM) with per-table norms and the
//               2x / 0x negative-count multipliers of the quirk; a small dense Adam/SGD kernel on the tower block.
// Parameter block W (flat fp32, module-registration order): per layer weight [out,in] + bias [out]; predict weight [2F] + bias.
//
// Rooflines: the tower is ~124 KFLOP per triple at F=32, L=2 (fwd+bwd, both items) against ~2.3 KB of embedding traffic:
// compute-bound on CUDA cores in the fp32 path (tower_dtype 0); with tower_dtype 1 the three GEMM call sites run on
// tcgen05 (umma_gemm.cuh) and the step becomes bound by streaming the fp32 activations (profiles/r01c).
#include "step.cuh"
#include "umma_gemm.cuh"
#include "neumf_fused.cuh"

namespace drb {

constexpr int kMaxLayers = 8;

struct NeumfDims {
    int U, I, F, L, D, mode;
    int n[kMaxLayers + 1];              // n[0] = 2D, n[l] = n[l-1]/2, n[L] = F
    long long w_off[kMaxLayers], b_off[kMaxLayers], wp_off, bp_off, nW;
    long long act_off[kMaxLayers + 1];  // offset of A_l inside the activation buffer, in units of R floats
    long long act_cols;                 // sum_l n[l]
};

// mode (config['model_name'], NeuMFRecommender.py:48-50,97-116,118-137): 0 'NeuMF' / 'NeuMF-pre' (predict over
// cat(GMF, tower) = 2F inputs), 1 'GMF' (predict over the GMF product, F inputs; the tower exists but is never run),
// 2 'MLP' (predict over the tower output, F inputs).  All four tables and every tower layer are parameters in every mode.
static bool make_dims(NeumfDims &d, int U, int I, int F, int L, int mode = 0)
{
    if (U <= 0 || I <= 0 || F <= 0 || L < 1 || L > kMaxLayers || (F % 4) != 0 || mode < 0 || mode > 2) return false;
    d.U = U; d.I = I; d.F = F; d.L = L; d.D = F << (L - 1); d.mode = mode;
    d.n[0] = 2 * d.D;
    long long o = 0, a = 0;
    for (int l = 0; l < L; ++l) {
        d.n[l + 1] = d.n[l] / 2;
        d.w_off[l] = o; o += (long long)d.n[l] * d.n[l + 1];
        d.b_off[l] = o; o += d.n[l + 1];
    }
    d.wp_off = o; o += (mode == 0 ? 2 : 1) * F;
    d.bp_off = o; o += 1;
    d.nW = o;
    for (int l = 0; l <= L; ++l) { d.act_off[l] = a; a += d.n[l]; }
    d.act_cols = a;
    return true;
}

struct NeumfWs {
    WsHeader *hdrG, *hdrM;       // phase-2 headers of the (UG,IG) and (UM,IM) table pairs
    double *red;                 // [16] batch reductions: bpr, l1[5], s2[5]  (UG_u, UM_u, IG_i, IM_i, IG_j)
    float *gUG, *gIG, *gUM, *gIM, *gW;
    unsigned *cntU;
    unsigned long long *cntI;
    float *mUG, *vUG, *mIG, *vIG, *mUM, *vUM, *mIM, *vIM, *mW, *vW;
    float *acts, *dA, *dB;       // activations [act_cols * R], two gradient ping-pong buffers [2D * R]
};

static size_t carve_neumf(void *base, const NeumfDims &d, int opt, long long max_rows, NeumfWs *w)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align256(bytes);
        return p;
    };
    NeumfWs t;
    t.hdrG = (WsHeader *)take(256);
    t.hdrM = (WsHeader *)take(256);
    t.red = (double *)take(16 * sizeof(double));
    const size_t uf = sizeof(float) * (size_t)d.U * d.F, itf = sizeof(float) * (size_t)d.I * d.F;
    const size_t ud = sizeof(float) * (size_t)d.U * d.D, itd = sizeof(float) * (size_t)d.I * d.D;
    const size_t wb = sizeof(float) * (size_t)d.nW;
    t.gUG = (float *)take(uf); t.gIG = (float *)take(itf); t.gUM = (float *)take(ud); t.gIM = (float *)take(itd);
    t.gW = (float *)take(wb);
    t.cntU = (unsigned *)take(sizeof(unsigned) * (size_t)d.U);
    t.cntI = (unsigned long long *)take(sizeof(unsigned long long) * (size_t)d.I);
    t.mUG = t.vUG = t.mIG = t.vIG = t.mUM = t.vUM = t.mIM = t.vIM = t.mW = t.vW = nullptr;
    if (opt == DRB_OPT_ADAM) {
        t.mUG = (float *)take(uf); t.vUG = (float *)take(uf); t.mIG = (float *)take(itf); t.vIG = (float *)take(itf);
        t.mUM = (float *)take(ud); t.vUM = (float *)take(ud); t.mIM = (float *)take(itd); t.vIM = (float *)take(itd);
        t.mW = (float *)take(wb); t.vW = (float *)take(wb);
    }
    t.acts = (float *)take(sizeof(float) * (size_t)d.act_cols * (size_t)max_rows);
    t.dA = (float *)take(sizeof(float) * (size_t)d.n[0] * (size_t)max_rows);
    t.dB = (float *)take(sizeof(float) * (size_t)d.n[0] * (size_t)max_rows);
    if (w) *w = t;
    return off;
}

// ------------------------------------------------------------------------------------------ generic fp32 GEMM
// C[M,N] (op)= opA(A)[M,K] * opB(B)[K,N];  64x64x16 tiles, 256 threads, 4x4 outputs per thread.
//   TA = false: A(m,k) = A[m*lda + k]      TA = true: A(m,k) = A[k*lda + m]
//   TB = false: B(k,n) = B[k*ldb + n]      TB = true: B(k,n) = B[n*ldb + k]
//   EPI 0: C = acc   1: C = relu(acc + bias[n])   2: C = acc * (ref(m,n) > 0)   3: atomicAdd(C, acc) (split-K over grid.z)
//   EPI 4: atomicAdd(C^T, acc): the product is accumulated into the transposed matrix C[n*ldc + m] (split-K)
template <bool TA, bool TB, int EPI>
__global__ void __launch_bounds__(256) sgemm_kernel(int M, int N, int K, const float *__restrict__ A, long long lda,
                                                    const float *__restrict__ B, long long ldb, float *__restrict__ C,
                                                    long long ldc, const float *__restrict__ bias,
                                                    const float *__restrict__ ref, long long ldref, int k_chunk,
                                                    float alpha)
{
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const long long m0 = (long long)blockIdx.x * 64;
    const int n0 = blockIdx.y * 64;
    const int kb = (EPI >= 3) ? blockIdx.z * k_chunk : 0;
    const int ke = (EPI >= 3) ? min(K, kb + k_chunk) : K;
    float acc[4][4] = {};
    for (int k0 = kb; k0 < ke; k0 += 16) {
        // load tiles: 16x64 each = 1024 elements, 4 per thread
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            int e = tid + q * 256;
            int kk, mm;
            if (TA) { kk = e >> 6; mm = e & 63; } else { mm = e >> 4; kk = e & 15; }
            long long m = m0 + mm;
            int k = k0 + kk;
            float v = 0.f;
            if (m < M && k < ke) v = TA ? __ldg(A + (long long)k * lda + m) : __ldg(A + m * lda + k);
            As[kk][mm] = v;
            int nn;
            if (TB) { nn = e >> 4; kk = e & 15; } else { kk = e >> 6; nn = e & 63; }
            int n = n0 + nn;
            k = k0 + kk;
            v = 0.f;
            if (n < N && k < ke) v = TB ? __ldg(B + (long long)n * ldb + k) : __ldg(B + (long long)k * ldb + n);
            Bs[kk][nn] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        long long m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            float v = acc[i][j];
            if (EPI == 1) { v += bias[n]; v = v > 0.f ? v : 0.f; }
            if (EPI == 2) { v = (ref[m * ldref + n] > 0.f) ? v * alpha : 0.f; }
            if (EPI == 3) atomicAdd(C + m * ldc + n, v);
            else if (EPI == 4) atomicAdd(C + (long long)n * ldc + m, v);   // transposed accumulate: C^T += acc
            else C[m * ldc + n] = v;
        }
    }
}

template <bool TA, bool TB, int EPI>
static int launch_sgemm(long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb, float *C,
                        long long ldc, const float *bias, const float *ref, long long ldref, cudaStream_t st, float alpha = 1.f)
{
    if (M <= 0 || N <= 0 || K <= 0) return DRB_OK;
    dim3 grid((unsigned)((M + 63) / 64), (unsigned)((N + 63) / 64), 1);
    int k_chunk = K;
    if (EPI >= 3) {   // split-K so that the tiny [out x in] result still fills the machine
        long long tiles = (long long)grid.x * grid.y;
        long long want = ((long long)sm_count() * 4 + tiles - 1) / tiles;          // chunks wanted for occupancy
        long long max_chunks = (K + 2047) / 2048;                                   // >= 2048 rows per chunk
        long long chunks = want < max_chunks ? want : max_chunks;
        if (chunks < 1) chunks = 1;
        k_chunk = (int)(((K + chunks - 1) / chunks + 15) / 16 * 16);
        grid.z = (unsigned)((K + k_chunk - 1) / k_chunk);
    }
    sgemm_kernel<TA, TB, EPI><<<grid, 256, 0, st>>>((int)M, N, K, A, lda, B, ldb, C, ldc, bias, ref, ldref, k_chunk, alpha);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

// dtype 0: fp32 CUDA cores (sgemm_kernel)   dtype 1: bf16 operands on tcgen05 tensor cores, fp32 accumulate in TMEM
template <bool TA, bool TB, int EPI>
static int launch_gemm(int dtype, long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb,
                       float *C, long long ldc, const float *bias, const float *ref, long long ldref, cudaStream_t st,
                       float alpha = 1.f)
{
    if (dtype == 1 && N <= kUmmaMaxN)
        return launch_umma_gemm<TA, TB, EPI>(M, N, K, A, lda, B, ldb, C, ldc, bias, ref, ldref, st, alpha);
    return launch_sgemm<TA, TB, EPI>(M, N, K, A, lda, B, ldb, C, ldc, bias, ref, ldref, st, alpha);
}

// ------------------------------------------------------------------------------------------ gather / head / scatter
// Dropout (NeuMFRecommender.py:61: nn.Dropout in front of every Linear, active in train mode).  The reference draws its
// masks from torch's global RNG; here they are counter-based: keep(layer, step, element) = Philox4x32-10(seed;
// element/4, layer, step) word (element%4) >= p * 2^32.  Counter-based masks can be regenerated in the backward pass
// (layer 0) instead of being stored.  Kept values are scaled by 1/(1-p) like torch.
// Parity mode: `bits[layer]` points at HOST-generated keep masks for this step -- the very tensors
// torch.empty(B, n_l).bernoulli_(1 - p) yields on the CPU generator, in the reference's draw order, bit-packed (bit e of
// the [2B, n_l] row-major mask; rows [0,B) from the pos forward, [B,2B) from the neg forward) -- and takes precedence.
struct Drop {
    float p, inv_keep;
    uint32_t k0, k1, step, thresh;
    const uint32_t *bits[kMaxLayers];
};

__device__ __forceinline__ float4 drop4(float4 v, const Drop &d, unsigned long long chunk, uint32_t layer)
{
    if (d.bits[0] != nullptr) {
        const uint32_t m = (__ldg(d.bits[layer] + (chunk >> 3)) >> ((unsigned)(chunk & 7ull) * 4u)) & 0xFu;
        v.x = (m & 1u) ? v.x * d.inv_keep : 0.f;
        v.y = (m & 2u) ? v.y * d.inv_keep : 0.f;
        v.z = (m & 4u) ? v.z * d.inv_keep : 0.f;
        v.w = (m & 8u) ? v.w * d.inv_keep : 0.f;
        return v;
    }
    uint32_t c[4] = {(uint32_t)chunk, (uint32_t)(chunk >> 32), layer, d.step};
    philox4x32(c, d.k0, d.k1);
    v.x = c[0] >= d.thresh ? v.x * d.inv_keep : 0.f;
    v.y = c[1] >= d.thresh ? v.y * d.inv_keep : 0.f;
    v.z = c[2] >= d.thresh ? v.z * d.inv_keep : 0.f;
    v.w = c[3] >= d.thresh ? v.w * d.inv_keep : 0.f;
    return v;
}

// in-place dropout of a hidden activation block (n4 float4 chunks)
__global__ void neumf_dropout_kernel(float *__restrict__ A, long long n4, Drop d, uint32_t layer)
{
    float4 *p = reinterpret_cast<float4 *>(A);
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += (long long)gridDim.x * blockDim.x)
        p[k] = drop4(p[k], d, (unsigned long long)k, layer);
}

// A_0[r, :] = cat(UM[u_r], IM[item_r]);  rows [0,B) use bi, rows [B,2B) use bj.   One thread per float4.
__global__ void neumf_gather_kernel(const float *__restrict__ UM, const float *__restrict__ IM, const int32_t *__restrict__ bu,
                                    const int32_t *__restrict__ bi, const int32_t *__restrict__ bj, long long B, int D,
                                    float *__restrict__ A0, Drop drop)
{
    const int d4 = D / 4;
    const long long total = 2 * B * 2 * d4;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        long long r = k / (2 * d4);
        int c = (int)(k - r * 2 * d4);
        long long t = r < B ? r : r - B;
        const float4 *src;
        if (c < d4) src = reinterpret_cast<const float4 *>(UM + (size_t)bu[t] * D) + c;
        else src = reinterpret_cast<const float4 *>(IM + (size_t)(r < B ? bi[t] : bj[t]) * D) + (c - d4);
        float4 v = __ldcg(src);
        if (drop.p > 0.f) v = drop4(v, drop, (unsigned long long)k, 0u);
        reinterpret_cast<float4 *>(A0 + (size_t)r * 2 * D)[c] = v;
    }
}

// inference variant: row r scores (users[r / per_user], item) with item = cands[r] or r % per_user
__global__ void neumf_gather_pairs_kernel(const float *__restrict__ UM, const float *__restrict__ IM,
                                          const int64_t *__restrict__ users, const int64_t *__restrict__ items,
                                          long long row0, long long rows, int per_user, int D, float *__restrict__ A0)
{
    const int d4 = D / 4;
    const long long total = rows * 2 * d4;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        long long r = k / (2 * d4);
        int c = (int)(k - r * 2 * d4);
        long long g = row0 + r;
        long long u = users[g / per_user];
        long long it = items ? items[g] : (g % per_user);
        const float4 *src = c < d4 ? reinterpret_cast<const float4 *>(UM + (size_t)u * D) + c
                                   : reinterpret_cast<const float4 *>(IM + (size_t)it * D) + (c - d4);
        reinterpret_cast<float4 *>(A0 + (size_t)r * 2 * D)[c] = __ldcg(src);
    }
}

// A group of W = min(32, next_pow2(F/4)) lanes per triple (4 triples per warp at F=32); float4 everywhere:
// 128-bit row loads, RED.ADD.F32x4 for the GMF-table gradients, 128-bit dZ_L stores.
// red[0] bpr, red[1..5] l1 of (UG_u, UM_u, IG_i, IM_i, IG_j), red[6..10] their squared sums.
__device__ __forceinline__ float4 ldcg4(const float *p) { return __ldcg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ float abs4(float4 v) { return fabsf(v.x) + fabsf(v.y) + fabsf(v.z) + fabsf(v.w); }
__device__ __forceinline__ float sq4(float4 v, float s) { return fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, s)))); }

__global__ void __launch_bounds__(256) neumf_head_kernel(const float *__restrict__ UG, const float *__restrict__ IG,
                                                         const float *__restrict__ UM, const float *__restrict__ IM,
                                                         const float *__restrict__ wp, const float *__restrict__ AL,
                                                         const int32_t *__restrict__ bu, const int32_t *__restrict__ bi,
                                                         const int32_t *__restrict__ bj, long long B, int F, int D, int has_reg,
                                                         int apply, int W, int mode, float *__restrict__ gUG, float *__restrict__ gIG,
                                                         float *__restrict__ gWp, float *__restrict__ dZL,
                                                         unsigned *__restrict__ cntU, unsigned long long *__restrict__ cntI,
                                                         double *__restrict__ red)
{
    extern __shared__ float s_gw[];                 // [2F + 1] CTA partial of the predict-layer gradient
    __shared__ double s_red[11];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int gpw = 32 / W, gl = lane % W, gw = lane / W;
    const int chunks = F / 4, dchunks = D / 4;
    // predict layer: mode 0 over cat(GMF, h) [2F], mode 1 over GMF [F], mode 2 over h [F]
    const bool use_g = mode != 2, use_h = mode != 1;
    const int pw = (mode == 0 ? 2 : 1) * F, hoff = mode == 0 ? F : 0;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = threadIdx.x; k < 2 * F + 1; k += blockDim.x) s_gw[k] = 0.f;
    if (threadIdx.x < 11) s_red[threadIdx.x] = 0.0;
    __syncthreads();
    float acc[11] = {};
    float4 gwa = make_float4(0.f, 0.f, 0.f, 0.f), gwb = gwa;   // predict-layer gradient partials of this lane's chunk
    const bool one_chunk = chunks <= W;                        // F <= 128: each lane owns at most one chunk
    const float bp = wp[pw];
    const long long groups = (long long)gridDim.x * nwarp * gpw;
    const long long g0 = ((long long)blockIdx.x * nwarp + warp) * gpw + gw;
    const long long rounds = (B + groups - 1) / groups;
    for (long long rd = 0; rd < rounds; ++rd) {
        const long long t = rd * groups + g0;
        const bool ok = t < B;
        const int u = ok ? bu[t] : 0, i = ok ? bi[t] : 0, j = ok ? bj[t] : 0;
        const float *ug = UG + (size_t)u * F, *igi = IG + (size_t)i * F, *igj = IG + (size_t)j * F;
        const float *hp = AL + (size_t)(ok ? t : 0) * F, *hn = AL + (size_t)(ok ? B + t : 0) * F;
        float sp = 0.f, sn = 0.f;
        for (int c = gl; c < chunks; c += W) {
            float4 a = ldcg4(ug + 4 * c), b = ldcg4(igi + 4 * c), d = ldcg4(igj + 4 * c);
            float4 w0 = use_g ? *reinterpret_cast<const float4 *>(wp + 4 * c) : z4;
            float4 w1 = use_h ? *reinterpret_cast<const float4 *>(wp + hoff + 4 * c) : z4;
            float4 h0 = use_h ? *reinterpret_cast<const float4 *>(hp + 4 * c) : z4, h1 = use_h ? *reinterpret_cast<const float4 *>(hn + 4 * c) : z4;
            sp = fmaf(w0.x, a.x * b.x, sp); sp = fmaf(w1.x, h0.x, sp); sn = fmaf(w0.x, a.x * d.x, sn); sn = fmaf(w1.x, h1.x, sn);
            sp = fmaf(w0.y, a.y * b.y, sp); sp = fmaf(w1.y, h0.y, sp); sn = fmaf(w0.y, a.y * d.y, sn); sn = fmaf(w1.y, h1.y, sn);
            sp = fmaf(w0.z, a.z * b.z, sp); sp = fmaf(w1.z, h0.z, sp); sn = fmaf(w0.z, a.z * d.z, sn); sn = fmaf(w1.z, h1.z, sn);
            sp = fmaf(w0.w, a.w * b.w, sp); sp = fmaf(w1.w, h0.w, sp); sn = fmaf(w0.w, a.w * d.w, sn); sn = fmaf(w1.w, h1.w, sn);
            if (has_reg && ok) {
                acc[1] += abs4(a); acc[6] = sq4(a, acc[6]);
                acc[3] += abs4(b); acc[8] = sq4(b, acc[8]);
                acc[5] += abs4(d); acc[10] = sq4(d, acc[10]);
            }
        }
        if (has_reg && ok) {
            const float *um = UM + (size_t)u * D, *imi = IM + (size_t)i * D;
            for (int c = gl; c < dchunks; c += W) {
                float4 a = ldcg4(um + 4 * c), b = ldcg4(imi + 4 * c);
                acc[2] += abs4(a); acc[7] = sq4(a, acc[7]);
                acc[4] += abs4(b); acc[9] = sq4(b, acc[9]);
            }
        }
        for (int off = W >> 1; off >= 1; off >>= 1) {
            sp += __shfl_xor_sync(0xffffffffu, sp, off);
            sn += __shfl_xor_sync(0xffffffffu, sn, off);
        }
        const float x = (sp + bp) - (sn + bp);
        const float sg = 1.f / (1.f + expf(-x));
        if (gl == 0 && ok) acc[0] += -logf(1e-10f + sg);
        const float c = -(sg * (1.f - sg)) / (1e-10f + sg);
        if (!apply || !ok) continue;
        for (int cc = gl; cc < chunks; cc += W) {
            float4 a = ldcg4(ug + 4 * cc), b = ldcg4(igi + 4 * cc), d = ldcg4(igj + 4 * cc);
            float4 w0 = use_g ? *reinterpret_cast<const float4 *>(wp + 4 * cc) : z4;
            float4 w1 = use_h ? *reinterpret_cast<const float4 *>(wp + hoff + 4 * cc) : z4;
            float4 h0 = use_h ? *reinterpret_cast<const float4 *>(hp + 4 * cc) : z4, h1 = use_h ? *reinterpret_cast<const float4 *>(hn + 4 * cc) : z4;
            // predict-layer weight gradient: dp * cat(GMF, h) summed over pos (+c) and neg (-c)
            float4 ga = make_float4(c * (a.x * b.x) - c * (a.x * d.x), c * (a.y * b.y) - c * (a.y * d.y),
                                    c * (a.z * b.z) - c * (a.z * d.z), c * (a.w * b.w) - c * (a.w * d.w));
            float4 gb = make_float4(c * h0.x - c * h1.x, c * h0.y - c * h1.y, c * h0.z - c * h1.z, c * h0.w - c * h1.w);
            if (one_chunk) {
                gwa.x += ga.x; gwa.y += ga.y; gwa.z += ga.z; gwa.w += ga.w;
                gwb.x += gb.x; gwb.y += gb.y; gwb.z += gb.z; gwb.w += gb.w;
            } else {
                if (use_g) { atomicAdd(&s_gw[4 * cc], ga.x); atomicAdd(&s_gw[4 * cc + 1], ga.y); atomicAdd(&s_gw[4 * cc + 2], ga.z); atomicAdd(&s_gw[4 * cc + 3], ga.w); }
                if (use_h) { atomicAdd(&s_gw[hoff + 4 * cc], gb.x); atomicAdd(&s_gw[hoff + 4 * cc + 1], gb.y); atomicAdd(&s_gw[hoff + 4 * cc + 2], gb.z); atomicAdd(&s_gw[hoff + 4 * cc + 3], gb.w); }
            }
            // GMF table gradients (one RED.ADD.F32x4 per row chunk)
            if (use_g) {
                Vec<4> v;
                v.v[0] = c * w0.x * b.x - c * w0.x * d.x; v.v[1] = c * w0.y * b.y - c * w0.y * d.y;
                v.v[2] = c * w0.z * b.z - c * w0.z * d.z; v.v[3] = c * w0.w * b.w - c * w0.w * d.w;
                red_row<4>(gUG + (size_t)u * F + 4 * cc, v);
                v.v[0] = c * w0.x * a.x; v.v[1] = c * w0.y * a.y; v.v[2] = c * w0.z * a.z; v.v[3] = c * w0.w * a.w;
                red_row<4>(gIG + (size_t)i * F + 4 * cc, v);
                v.v[0] = -v.v[0]; v.v[1] = -v.v[1]; v.v[2] = -v.v[2]; v.v[3] = -v.v[3];
                red_row<4>(gIG + (size_t)j * F + 4 * cc, v);
            }
            if (use_h) {
                // dZ_L = dp * w1 * relu'(h)
                *reinterpret_cast<float4 *>(dZL + (size_t)t * F + 4 * cc) =
                    make_float4(h0.x > 0.f ? c * w1.x : 0.f, h0.y > 0.f ? c * w1.y : 0.f, h0.z > 0.f ? c * w1.z : 0.f, h0.w > 0.f ? c * w1.w : 0.f);
                *reinterpret_cast<float4 *>(dZL + (size_t)(B + t) * F + 4 * cc) =
                    make_float4(h1.x > 0.f ? -c * w1.x : 0.f, h1.y > 0.f ? -c * w1.y : 0.f, h1.z > 0.f ? -c * w1.z : 0.f, h1.w > 0.f ? -c * w1.w : 0.f);
            }
        }
        if (gl == 0) {
            red_add_u32(cntU + u, 1u);
            red_add_u64(cntI + i, 1ull);
            red_add_u64(cntI + j, 1ull << 32);
        }
    }
    if (apply && one_chunk && gl < chunks) {
        if (use_g) { atomicAdd(&s_gw[4 * gl], gwa.x); atomicAdd(&s_gw[4 * gl + 1], gwa.y); atomicAdd(&s_gw[4 * gl + 2], gwa.z); atomicAdd(&s_gw[4 * gl + 3], gwa.w); }
        if (use_h) { atomicAdd(&s_gw[hoff + 4 * gl], gwb.x); atomicAdd(&s_gw[hoff + 4 * gl + 1], gwb.y); atomicAdd(&s_gw[hoff + 4 * gl + 2], gwb.z); atomicAdd(&s_gw[hoff + 4 * gl + 3], gwb.w); }
    }
    // block reduction of the scalars
    const int nv = has_reg ? 11 : 1;
    for (int k = 0; k < nv; ++k) {
        float v = acc[k];
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if (lane == 0) atomicAdd(&s_red[k], (double)v);
    }
    __syncthreads();
    if (threadIdx.x < nv && s_red[threadIdx.x] != 0.0) atomicAdd(red + threadIdx.x, s_red[threadIdx.x]);
    if (apply)
        for (int k = threadIdx.x; k < pw; k += blockDim.x)
            if (s_gw[k] != 0.f) atomicAdd(gWp + k, s_gw[k]);
    // the bias gradient of the predict layer is sum(+c) + sum(-c) == 0 exactly for a pairwise loss
}

// gb[n] += sum_m dZ[m, n]      (coalesced: consecutive threads read consecutive columns of one row)
__global__ void __launch_bounds__(256) colsum_kernel(const float *__restrict__ dZ, long long M, int N, float *__restrict__ gb)
{
    __shared__ float s_part[256];
    const int rows_per_pass = 256 / N > 0 ? 256 / N : 1;       // N <= 256
    const int tr = threadIdx.x / N, tn = threadIdx.x % N;
    float s = 0.f;
    if (tr < rows_per_pass)
        for (long long m = (long long)blockIdx.x * rows_per_pass + tr; m < M; m += (long long)gridDim.x * rows_per_pass)
            s += dZ[m * N + tn];
    s_part[threadIdx.x] = (tr < rows_per_pass) ? s : 0.f;
    __syncthreads();
    if (threadIdx.x < N) {
        float t = 0.f;
        for (int q = 0; q < rows_per_pass; ++q) t += s_part[q * N + threadIdx.x];
        if (t != 0.f) atomicAdd(gb + threadIdx.x, t);
    }
}

// gUM[u] += dA0[t,:D] + dA0[B+t,:D];  gIM[i] += dA0[t,D:];  gIM[j] += dA0[B+t,D:]      (RED.ADD.F32x4)
__global__ void neumf_scatter_kernel(const float *__restrict__ dA0, const int32_t *__restrict__ bu,
                                     const int32_t *__restrict__ bi, const int32_t *__restrict__ bj, long long B, int D,
                                     float *__restrict__ gUM, float *__restrict__ gIM, Drop drop)
{
    const int d4 = D / 4;
    const long long total = B * d4;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        long long t = k / d4;
        int c = (int)(k - t * d4);
        const float4 *rp = reinterpret_cast<const float4 *>(dA0 + (size_t)t * 2 * D);
        const float4 *rn = reinterpret_cast<const float4 *>(dA0 + (size_t)(B + t) * 2 * D);
        float4 up = rp[c], un = rn[c], ip = rp[d4 + c], in_ = rn[d4 + c];
        if (drop.p > 0.f) {   // d(A_0) = d(A_0') * mask_0 / (1-p): same counters as the gather (chunk = row * 2*d4 + col)
            const unsigned long long cp = (unsigned long long)t * 2 * d4, cn = (unsigned long long)(B + t) * 2 * d4;
            up = drop4(up, drop, cp + c, 0u); un = drop4(un, drop, cn + c, 0u);
            ip = drop4(ip, drop, cp + d4 + c, 0u); in_ = drop4(in_, drop, cn + d4 + c, 0u);
        }
        Vec<4> v;
        v.v[0] = up.x + un.x; v.v[1] = up.y + un.y; v.v[2] = up.z + un.z; v.v[3] = up.w + un.w;
        red_row<4>(gUM + (size_t)bu[t] * D + c * 4, v);
        v.v[0] = ip.x; v.v[1] = ip.y; v.v[2] = ip.z; v.v[3] = ip.w;
        red_row<4>(gIM + (size_t)bi[t] * D + c * 4, v);
        v.v[0] = in_.x; v.v[1] = in_.y; v.v[2] = in_.z; v.v[3] = in_.w;
        red_row<4>(gIM + (size_t)bj[t] * D + c * 4, v);
    }
}

// Assemble the fp32 loss in the reference's order (NeuMFRecommender.py:154-167), publish it, and prime the two
// phase-2 headers (norms per table pair; NaN -> sticky status so that nothing is applied).
__global__ void neumf_finalize_kernel(const double *__restrict__ red, float reg1, float reg2, WsHeader *hG, WsHeader *hM,
                                      double *__restrict__ loss_out, long long step)
{
    const double bpr = red[0];
    const double *l1 = red + 1, *s2 = red + 6;     // 0 UG_u, 1 UM_u, 2 IG_i, 3 IM_i, 4 IG_j
    double nr[5];
    for (int q = 0; q < 5; ++q) nr[q] = sqrt(s2[q]);
    float loss = (float)bpr;
    loss += reg1 * ((float)l1[2] + (float)l1[4]);
    loss += reg1 * ((float)l1[3] + (float)l1[4]);
    loss += reg2 * ((float)nr[2] + (float)nr[4]);
    loss += reg2 * ((float)nr[3] + (float)nr[4]);
    loss += reg1 * (float)l1[0];
    loss += reg1 * (float)l1[1];
    loss += reg2 * (float)nr[0];
    loss += reg2 * (float)nr[1];
    *loss_out = (double)loss;
    const bool bad = isnan(loss);
    // phase 2 reads acc[0] = {bpr, l1u, l1i, l1j, s2u, s2i, s2j}; only the squared sums matter for the update
    double *g = hG->acc[0], *m = hM->acc[0];
    g[0] = bad ? (double)loss : 0.0; g[1] = g[2] = g[3] = 0.0; g[4] = s2[0]; g[5] = s2[2]; g[6] = s2[4];
    m[0] = bad ? (double)loss : 0.0; m[1] = m[2] = m[3] = 0.0; m[4] = s2[1]; m[5] = s2[3]; m[6] = 0.0;
    if (bad) {
        hG->status = DRB_ERR_NAN_LOSS; hG->nan_step = step;
        hM->status = DRB_ERR_NAN_LOSS; hM->nan_step = step;
    }
}

// scores[r] = wp . cat(UG[u]*IG[item], A_L[r]) + bp      (inference head)
__global__ void neumf_score_kernel(const float *__restrict__ UG, const float *__restrict__ IG, const float *__restrict__ wp,
                                   const float *__restrict__ AL, const int64_t *__restrict__ users,
                                   const int64_t *__restrict__ items, long long row0, long long rows, int per_user, int F,
                                   int mode, float *__restrict__ scores)
{
    const bool use_g = mode != 2, use_h = mode != 1;
    const int pw = (mode == 0 ? 2 : 1) * F, hoff = mode == 0 ? F : 0;
    const int lane = threadIdx.x & 31;
    long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < rows; r += nw) {
        long long g = row0 + r;
        long long u = users[g / per_user];
        long long it = items ? items[g] : (g % per_user);
        float s = 0.f;
        for (int f = lane; f < F; f += 32) {
            if (use_g) s = fmaf(wp[f], __ldcg(UG + (size_t)u * F + f) * __ldcg(IG + (size_t)it * F + f), s);
            if (use_h) s = fmaf(wp[hoff + f], AL[(size_t)r * F + f], s);
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane == 0) scores[g] = s + wp[pw];
    }
}

// ---- the tower's GEMM dispatcher for the other dense-layer models (ngcf.cu): plain entry points, see gemm.cuh
int gemm_nt(int dtype, long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb, float *C,
            long long ldc, cudaStream_t st)
{
    return launch_gemm<false, true, 0>(dtype, M, N, K, A, lda, B, ldb, C, ldc, nullptr, nullptr, 0, st);
}
int gemm_nn(int dtype, long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb, float *C,
            long long ldc, cudaStream_t st)
{
    return launch_gemm<false, false, 0>(dtype, M, N, K, A, lda, B, ldb, C, ldc, nullptr, nullptr, 0, st);
}
int gemm_tn_acc_t(int dtype, long long M, int N, int K, const float *A, long long lda, const float *B, long long ldb, float *C,
                  long long ldc, cudaStream_t st)
{
    return launch_gemm<true, false, 4>(dtype, M, N, K, A, lda, B, ldb, C, ldc, nullptr, nullptr, 0, st);
}
int colsum_acc(const float *dZ, long long M, int N, float *gb, cudaStream_t st)
{
    DRB_REQUIRE(N <= 256, "colsum: N=%d exceeds 256", N);
    colsum_kernel<<<sm_count() * 4, 256, 0, st>>>(dZ, M, N, gb);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

// dense optimiser step on a flat block (SGD, or torch.optim.Adam's single-tensor rule); clears the gradient
__global__ void dense_update_kernel(float *__restrict__ W, float *__restrict__ g, float *__restrict__ m, float *__restrict__ v,
                                    long long n, float lr, int opt, float beta1, float beta2, float eps, float step_size,
                                    float bc2_sqrt, const WsHeader *hdr)
{
    if (hdr->status != 0) return;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const float gk = g[k];
        g[k] = 0.f;
        if (opt == DRB_OPT_SGD) {
            W[k] = W[k] - lr * gk;
        } else {
            float mm = m[k], vv = v[k];
            mm = mm + (gk - mm) * (1.f - beta1);
            vv = vv * beta2 + (1.f - beta2) * gk * gk;
            W[k] = W[k] - step_size * (mm / (sqrtf(vv) / bc2_sqrt + eps));
            m[k] = mm; v[k] = vv;
        }
    }
}
int dense_update(float *W, float *g, float *m, float *v, long long n, const drb_hyper *h, long long adam_step, const WsHeader *hdr,
                 cudaStream_t st)
{
    const double t = (double)(adam_step + 1);
    const float step_size = (float)((double)h->lr / (1.0 - pow((double)h->beta1, t)));
    const float bc2_sqrt = (float)sqrt(1.0 - pow((double)h->beta2, t));
    dense_update_kernel<<<grid_size(n, 256), 256, 0, st>>>(W, g, m, v, n, h->lr, h->opt, h->beta1, h->beta2, h->eps, step_size,
                                                           bc2_sqrt, hdr);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

// tower forward on `rows` rows already gathered into acts' A_0 block
static int tower_forward(const NeumfDims &d, const float *W, float *acts, long long R, long long rows, int dtype,
                         const Drop &drop, cudaStream_t st)
{
    for (int l = 0; l < d.L; ++l) {
        const float *in = acts + d.act_off[l] * R;
        float *out = acts + d.act_off[l + 1] * R;
        int rc = launch_gemm<false, true, 1>(dtype, rows, d.n[l + 1], d.n[l], in, d.n[l], W + d.w_off[l], d.n[l], out,
                                             d.n[l + 1], W + d.b_off[l], nullptr, 0, st);
        if (rc != DRB_OK) return rc;
        if (drop.p > 0.f && l + 1 < d.L) {   // the next Linear sees dropout(relu(z_l)); the tower output is not dropped
            long long n4 = rows * d.n[l + 1] / 4;
            neumf_dropout_kernel<<<grid_size(n4, 256), 256, 0, st>>>(out, n4, drop, (uint32_t)(l + 1));
            DRB_CUDA(cudaGetLastError());
        }
    }
    return DRB_OK;
}

}  // namespace drb

using namespace drb;

extern "C" int64_t drb_neumf_param_count(int32_t F, int32_t L, int32_t mode)
{
    NeumfDims d;
    if (!make_dims(d, 1, 1, F, L, mode)) return -1;
    return d.nW;
}

// words (uint32) of host-generated dropout keep-masks one step of `batch` triples consumes: layer l's [2*batch, n_l] mask
// bit-packed and padded to a word, layers in order (n_0 = 2D, n_l = n_{l-1}/2)
extern "C" int64_t drb_neumf_mask_words(int32_t F, int32_t L, int64_t batch)
{
    NeumfDims d;
    if (!make_dims(d, 1, 1, F, L)) return -1;
    int64_t w = 0;
    for (int l = 0; l < L; ++l) w += (2 * batch * d.n[l] + 31) / 32;
    return w;
}

extern "C" size_t drb_neumf_workspace_bytes(int32_t U, int32_t I, int32_t F, int32_t L, int32_t opt, int64_t max_rows)
{
    NeumfDims d;
    if (!make_dims(d, U, I, F, L)) return 0;      // mode 0 has the largest parameter block: one layout for every mode
    return carve_neumf(nullptr, d, opt, max_rows, nullptr);
}

extern "C" int drb_neumf_workspace_init(void *d_ws, int32_t U, int32_t I, int32_t F, int32_t L, int32_t opt,
                                        int64_t max_rows, void *stream)
{
    NeumfDims d;
    DRB_REQUIRE(d_ws && make_dims(d, U, I, F, L), "neumf_workspace_init: bad arguments (factors must be a multiple of 4)");
    NeumfWs w;
    carve_neumf(d_ws, d, opt, max_rows, &w);
    // zero everything except the (large) activation scratch
    size_t head = (size_t)((char *)w.acts - (char *)d_ws);
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, head, (cudaStream_t)stream));
    return DRB_OK;
}

// n_steps synchronous NeuMF+BPR steps (apply != 0) or the loss of one batch (apply == 0).
extern "C" int drb_neumf_bpr_train_steps(float *d_UG, float *d_IG, float *d_UM, float *d_IM, float *d_W, void *d_ws,
                                         int32_t U, int32_t I, int32_t F, int32_t L, int64_t max_rows,
                                         const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n,
                                         int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *h,
                                         int64_t adam_step0, int32_t apply, int32_t tower_dtype, float dropout,
                                         uint64_t dropout_seed, const uint32_t *d_drop_masks, int32_t mode,
                                         double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream)
{
    NeumfDims d, dlay;
    DRB_REQUIRE(tower_dtype >= 0 && tower_dtype <= 2,
                "neumf: tower_dtype must be 0 (fp32), 1 (bf16 tcgen05, layer-wise) or 2 (bf16 tcgen05, fused per tile)");
    DRB_REQUIRE(dropout >= 0.f && dropout < 1.f, "neumf: dropout must be in [0, 1)");
    const bool fused = tower_dtype == 2 && neumf_fused_supported(F, L, mode, dropout);
    if (tower_dtype == 2 && !fused) tower_dtype = 1;      // shapes outside the fused kernel: same numerics class, layer-wise
    DRB_REQUIRE(make_dims(d, U, I, F, L, mode) && make_dims(dlay, U, I, F, L, 0),
                "neumf: bad dims (factors must be a positive multiple of 4, 1 <= num_layers <= 8, mode 0..2)");
    DRB_REQUIRE(d_UG && d_IG && d_UM && d_IM && d_W && d_ws && d_bu && d_bi && d_bj && h && d_step_loss, "neumf: null argument");
    DRB_REQUIRE(batch > 0 && 2 * batch <= max_rows, "neumf: batch %lld needs 2*batch <= max_rows=%lld", (long long)batch,
                (long long)max_rows);
    DRB_REQUIRE(n_steps == 0 || (first_step + n_steps - 1) * batch < n, "neumf: steps exceed %lld triples", (long long)n);
    DRB_REQUIRE(h->opt == DRB_OPT_SGD || h->opt == DRB_OPT_ADAM, "unknown optimizer id %d", h->opt);
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    NeumfWs w;
    carve_neumf(d_ws, dlay, h->opt, max_rows, &w);
    const int has_reg = (h->reg_1 != 0.f) || (h->reg_2 != 0.f);
    const bool use_tower = mode != 1;
    const int64_t mask_words = d_drop_masks ? drb_neumf_mask_words(F, L, batch) : 0;
    DRB_CUDA(cudaMemsetAsync(w.hdrG, 0, 512, st));            // both headers: clear a stale NaN flag
    for (int64_t s = 0; s < n_steps; ++s) {
        const int64_t base = (first_step + s) * batch, B = (n - base < batch) ? n - base : batch;
        const long long R = 2 * B;
        const int32_t *bu = d_bu + base, *bi = d_bi + base, *bj = d_bj + base;
        DRB_CUDA(cudaMemsetAsync(w.red, 0, 16 * sizeof(double), st));
        Drop drop;
        drop.p = dropout; drop.inv_keep = 1.f / (1.f - dropout);
        drop.k0 = (uint32_t)dropout_seed; drop.k1 = (uint32_t)(dropout_seed >> 32);
        drop.step = (uint32_t)(adam_step0 + s);
        drop.thresh = (uint32_t)fmin(4294967295.0, (double)dropout * 4294967296.0);
        for (int l = 0; l < kMaxLayers; ++l) drop.bits[l] = nullptr;
        if (d_drop_masks && dropout > 0.f) {                  // parity mode: this step's host-generated masks, per layer
            DRB_REQUIRE(B == batch, "neumf: host dropout masks need full batches (n must be a multiple of batch)");
            const uint32_t *mp = d_drop_masks + (size_t)s * (size_t)mask_words;
            for (int l = 0; l < d.L; ++l) {
                drop.bits[l] = mp;
                mp += (2 * batch * d.n[l] + 31) / 32;
            }
        }
        int rc = DRB_OK;
        if (fused) {
            // one persistent kernel: gather, both layers, head, all four backward products, scatter (neumf_fused.cuh)
            FusedParams fp;
            fp.UG = d_UG; fp.IG = d_IG; fp.UM = d_UM; fp.IM = d_IM; fp.W = d_W;
            fp.bu = bu; fp.bi = bi; fp.bj = bj; fp.B = B;
            fp.gUG = w.gUG; fp.gIG = w.gIG; fp.gUM = w.gUM; fp.gIM = w.gIM; fp.gW = w.gW;
            fp.cntU = w.cntU; fp.cntI = w.cntI; fp.red = w.red; fp.has_reg = has_reg; fp.apply = apply ? 1 : 0;
            rc = launch_neumf_fused(F, fp, st);
            if (rc != DRB_OK) return rc;
            neumf_finalize_kernel<<<1, 1, 0, st>>>(w.red, h->reg_1, h->reg_2, w.hdrG, w.hdrM, d_step_loss + s, first_step + s);
            DRB_CUDA(cudaGetLastError());
            if (!apply) break;
        }
        // forward
        if (use_tower && !fused) {
            neumf_gather_kernel<<<grid_size(R * 2 * (d.D / 4), 256), 256, 0, st>>>(d_UM, d_IM, bu, bi, bj, B, d.D, w.acts, drop);
            DRB_CUDA(cudaGetLastError());
            rc = tower_forward(d, d_W, w.acts, R, R, tower_dtype, drop, st);
            if (rc != DRB_OK) return rc;
        }
        const float *AL = w.acts + d.act_off[d.L] * R;
        float *dZ = w.dA;                                        // dZ_L [R, F]
        if (!fused) {
            int hw = 1;
            while (hw < F / 4 && hw < 32) hw <<= 1;              // lanes per triple in the head kernel
            neumf_head_kernel<<<grid_size(B, 8 * (32 / hw), 8), 256, sizeof(float) * (2 * F + 1), st>>>(
                d_UG, d_IG, d_UM, d_IM, d_W + d.wp_off, AL, bu, bi, bj, B, F, d.D, has_reg, apply ? 1 : 0, hw, mode, w.gUG, w.gIG,
                w.gW + d.wp_off, dZ, w.cntU, w.cntI, w.red);
            DRB_CUDA(cudaGetLastError());
            neumf_finalize_kernel<<<1, 1, 0, st>>>(w.red, h->reg_1, h->reg_2, w.hdrG, w.hdrM, d_step_loss + s, first_step + s);
            DRB_CUDA(cudaGetLastError());
            if (!apply) break;
        }
        // tower backward ('GMF': the tower takes no part in the prediction, its parameters have no gradient)
        float *cur = w.dA, *nxt = w.dB;
        for (int l = d.L - 1; l >= 0 && use_tower && !fused; --l) {
            const float *Aprev = w.acts + d.act_off[l] * R;
            // gW_l[out,in] += dZ^T A_{l-1}, computed as (A_{l-1}^T dZ)^T: the wide dimension (in) fills the 128-row MMA tile
            // and the narrow one (out) becomes N, so the TMEM footprint per CTA is small and more CTAs overlap
            // (split-K over the R rows; transposed atomic accumulate into gW_l)
            rc = launch_gemm<true, false, 4>(tower_dtype, d.n[l], d.n[l + 1], (int)R, Aprev, d.n[l], cur, d.n[l + 1], w.gW + d.w_off[l],
                                              d.n[l], nullptr, nullptr, 0, st);
            if (rc != DRB_OK) return rc;
            colsum_kernel<<<sm_count() * 4, 256, 0, st>>>(cur, R, d.n[l + 1], w.gW + d.b_off[l]);
            DRB_CUDA(cudaGetLastError());
            // dA_{l-1} = dZ W_l, masked by relu'(A_{l-1}) for hidden layers
            if (l > 0)
                rc = launch_gemm<false, false, 2>(tower_dtype, R, d.n[l], d.n[l + 1], cur, d.n[l + 1], d_W + d.w_off[l], d.n[l], nxt,
                                                   d.n[l], nullptr, Aprev, d.n[l], st, drop.inv_keep);
            else
                rc = launch_gemm<false, false, 0>(tower_dtype, R, d.n[l], d.n[l + 1], cur, d.n[l + 1], d_W + d.w_off[l], d.n[l], nxt,
                                                   d.n[l], nullptr, nullptr, 0, st);
            if (rc != DRB_OK) return rc;
            float *t = cur; cur = nxt; nxt = t;
        }
        if (use_tower && !fused) {
            neumf_scatter_kernel<<<grid_size(B * (d.D / 4), 256), 256, 0, st>>>(cur, bu, bi, bj, B, d.D, w.gUM, w.gIM, drop);
            DRB_CUDA(cudaGetLastError());
        }
        // apply: table pairs through the MF dense sweep, tower block through the small dense kernel
        StepParams p = split_step(h, U, I, bu, bi, bj, B, adam_step0 + s, w.red + 12);   // scratch: finalize wrote the loss
        p.phases = 2;
        p.ws.cntU = w.cntU; p.ws.cntI = w.cntI;
        // (UG, IG): negative occurrences weigh 2x (lines :157 and :158 both add |IG_j|)
        p.P = d_UG; p.Q = d_IG; p.F = F; p.ws.hdr = w.hdrG; p.ws.gP = w.gUG; p.ws.gQ = w.gIG;
        p.ws.mP = w.mUG; p.ws.vP = w.vUG; p.ws.mQ = w.mIG; p.ws.vQ = w.vIG; p.neg_mult = 2.f; p.keep_counts = 1;
        rc = launch_steps(p, st, true);
        if (rc != DRB_OK) return rc;
        // (UM, IM): the MLP item table is never regularised on the negative side
        p.P = d_UM; p.Q = d_IM; p.F = d.D; p.ws.hdr = w.hdrM; p.ws.gP = w.gUM; p.ws.gQ = w.gIM;
        p.ws.mP = w.mUM; p.ws.vP = w.vUM; p.ws.mQ = w.mIM; p.ws.vQ = w.vIM; p.neg_mult = 0.f; p.keep_counts = 0;
        rc = launch_steps(p, st, true);
        if (rc == DRB_OK) rc = dense_update(d_W, w.gW, w.mW, w.vW, d.nW, h, adam_step0 + s, w.hdrG, st);
        if (rc != DRB_OK) return rc;
    }
    if (sync_and_check) return check_nan(w.hdrG, st, nan_step);
    return DRB_OK;
}

// scores[n_users * per_user] for (users[r / per_user], items[r]) pairs (items == NULL: every item id 0..per_user-1)
extern "C" int drb_neumf_scores(const float *d_UG, const float *d_IG, const float *d_UM, const float *d_IM, const float *d_W,
                                void *d_ws, int32_t U, int32_t I, int32_t F, int32_t L, int32_t opt, int64_t max_rows,
                                const int64_t *d_users, int64_t n_users, const int64_t *d_items, int32_t per_user,
                                int32_t tower_dtype, int32_t mode, float *d_scores, void *stream)
{
    NeumfDims d, dlay;
    DRB_REQUIRE(make_dims(d, U, I, F, L, mode) && make_dims(dlay, U, I, F, L, 0), "neumf_scores: bad dims");
    DRB_REQUIRE(d_UG && d_IG && d_UM && d_IM && d_W && d_ws && d_users && d_scores && per_user > 0 && max_rows > 0,
                "neumf_scores: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    NeumfWs w;
    carve_neumf(d_ws, dlay, opt, max_rows, &w);   // same layout as training: only the dA/dB scratch is touched here
    const long long total = (long long)n_users * per_user;
    for (long long row0 = 0; row0 < total; row0 += max_rows) {
        long long rows = total - row0 < max_rows ? total - row0 : max_rows;
        if (mode != 1) {
            neumf_gather_pairs_kernel<<<grid_size(rows * 2 * (d.D / 4), 256), 256, 0, st>>>(d_UM, d_IM, d_users, d_items, row0, rows,
                                                                                            per_user, d.D, w.dA);
            DRB_CUDA(cudaGetLastError());
        }
        // use dA as A_0 and dB as ping-pong for the hidden layers (independent of the optimiser layout)
        const float *in = w.dA;
        float *bufs[2] = {w.dB, w.dA};
        for (int l = 0; l < d.L && mode != 1; ++l) {
            float *out = bufs[l & 1];
            int rc = launch_gemm<false, true, 1>(tower_dtype, rows, d.n[l + 1], d.n[l], in, d.n[l], d_W + d.w_off[l], d.n[l],
                                                 out, d.n[l + 1], d_W + d.b_off[l], nullptr, 0, st);
            if (rc != DRB_OK) return rc;
            in = out;
        }
        neumf_score_kernel<<<grid_size(rows * 32, 256), 256, 0, st>>>(d_UG, d_IG, d_W + d.wp_off, in, d_users, d_items, row0, rows,
                                                                      per_user, F, mode, d_scores);
        DRB_CUDA(cudaGetLastError());
    }
    return DRB_OK;
}

// Test hook: C (op)= opA(A) opB(B) through the tower's GEMM dispatcher.  variant 0: NT + bias + ReLU (forward),
// 1: NN + ReLU mask (input gradient), 2: NN plain, 3: TN split-K accumulate (weight gradient).  dtype as tower_dtype.
extern "C" int drb_gemm_test(int32_t variant, int32_t dtype, int64_t M, int32_t N, int32_t K, const float *d_A, int64_t lda,
                             const float *d_B, int64_t ldb, float *d_C, int64_t ldc, const float *d_bias, const float *d_ref,
                             int64_t ldref, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    switch (variant) {
    case 0: return launch_gemm<false, true, 1>(dtype, M, N, K, d_A, lda, d_B, ldb, d_C, ldc, d_bias, nullptr, 0, st);
    case 1: return launch_gemm<false, false, 2>(dtype, M, N, K, d_A, lda, d_B, ldb, d_C, ldc, nullptr, d_ref, ldref, st);
    case 2: return launch_gemm<false, false, 0>(dtype, M, N, K, d_A, lda, d_B, ldb, d_C, ldc, nullptr, nullptr, 0, st);
    case 3: return launch_gemm<true, false, 3>(dtype, M, N, K, d_A, lda, d_B, ldb, d_C, ldc, nullptr, nullptr, 0, st);
    case 4: return launch_gemm<true, false, 4>(dtype, M, N, K, d_A, lda, d_B, ldb, d_C, ldc, nullptr, nullptr, 0, st);
    }
    DRB_REQUIRE(false, "gemm_test: unknown variant %d", variant);
}
