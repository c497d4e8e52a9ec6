// vae.cu -- Multi-VAE (VAECF) on the B200 path.
//
// Stands behind daisy/model/VAECFRecommender.py:
//   forward   :79-90   h = F.normalize(R) (row L2, eps 1e-12) -> F.dropout(p) -> encoder (item_num -> h_1 .. h_L -> latent_dim,
//                      Tanh between layers) -> mu = h[:, :lat/2], logvar = h[:, ceil(lat/2):] -> z = eps * exp(0.5 logvar) + mu
//                      (train) or mu (eval) -> decoder (lat/2 -> h_L .. h_1 -> item_num, Tanh between layers)
//   calc_loss :92-110  CE = -(log_softmax(logits) * R).sum(1).mean() on the UN-normalised R, KL = -0.5 mean(sum(1 + lv - mu^2
//                      - e^lv)) * anneal, anneal = min(cap, update / total_anneal_steps)
//   backward + optimizer.step (SGD or Adam over every parameter)
//
// R stays sparse: a user's ratings are a CSR row (row_ptr, col, val) built once from the padded history.  The first
// encoder Linear is a sparse product over the row's nonzeros (its weight is stored transposed, [item_num, h_1], so an
// item's row is contiguous), and so is its weight gradient.  The decoder's output layer is the wide one: its logits are
// kept item-major, L^T [item_num, B], so that the item dimension is the M dimension of every wide GEMM (tensor-core path
// with tower_dtype 1) and B is sliced into panels of at most kUmmaMaxN columns.  Softmax cross-entropy runs over L^T in
// two passes (per-chunk online max / sum-exp, then the combined log-sum-exp) and writes dL = softmax * S_b / B - R / B in
// place, S_b = sum of the row's ratings; the decoder output-bias gradient is the row sum of dL^T.
//
// Parameter block N (flat fp32, module registration order): encoder.0 W^T [I, e1], b [e1], encoder.2 W [e2, e1], b, ...,
// decoder.0 W [d1, lat/2], b, ..., decoder.2L W [I, h_1], b [I]; each weight and bias is padded with zeros to a multiple of
// 4 floats, so every one starts 16-byte aligned (the padding has no gradient and never moves).  One dense_update() moves
// the whole block per step.
#include "gemm.cuh"
#include "step.cuh"

namespace drb {

constexpr int kVaeMaxL = 8;
constexpr int kVaePanel = 256;                 // B columns per wide GEMM (kUmmaMaxN)

struct VaeDims {
    int I, L, lat, half, lvo, ne;             // ne = L + 1 Linear layers per side; lvo = ceil(lat / 2)
    int e[kVaeMaxL + 2], d[kVaeMaxL + 2];     // encoder widths [I, h_1..h_L, lat], decoder widths [lat/2, h_L..h_1, I]
    long long oEW[kVaeMaxL + 1], oEB[kVaeMaxL + 1], oDW[kVaeMaxL + 1], oDB[kVaeMaxL + 1], nN;
    int maxw;                                 // widest hidden / latent activation (everything but I)
};

static bool vae_dims(VaeDims &v, int I, const int32_t *hidden, int L, int lat)
{
    if (I <= 0 || L < 0 || L > kVaeMaxL || lat < 2 || (L > 0 && !hidden)) return false;
    v.I = I; v.L = L; v.lat = lat; v.half = lat / 2; v.lvo = lat - lat / 2; v.ne = L + 1;
    v.e[0] = I;
    for (int k = 0; k < L; ++k) {
        if (hidden[k] <= 0) return false;
        v.e[k + 1] = hidden[k];
    }
    v.e[L + 1] = lat;
    v.d[0] = v.half;
    for (int k = 1; k <= L; ++k) v.d[k] = v.e[L + 1 - k];
    v.d[L + 1] = I;
    // every weight and bias starts on a 4-float (16-byte) boundary: the bf16 GEMM stages its operands with float4 loads
    auto pad4 = [](long long x) { return (x + 3) & ~3ll; };
    long long o = 0;
    for (int k = 0; k < v.ne; ++k) {
        v.oEW[k] = o; o = pad4(o + (long long)v.e[k] * v.e[k + 1]);
        v.oEB[k] = o; o = pad4(o + v.e[k + 1]);
    }
    for (int k = 0; k < v.ne; ++k) {
        v.oDW[k] = o; o = pad4(o + (long long)v.d[k] * v.d[k + 1]);
        v.oDB[k] = o; o = pad4(o + v.d[k + 1]);
    }
    v.nN = o;
    v.maxw = lat;
    for (int k = 1; k <= L; ++k) v.maxw = v.e[k] > v.maxw ? v.e[k] : v.maxw;
    return true;
}

struct VaeWs {
    WsHeader *hdr;
    float *gN, *mN, *vN;                      // gradient accumulator and Adam state of the parameter block
    float *denom, *S, *lse;                   // [R]: max(||r||, 1e-12), sum r, log-sum-exp of the logits
    float *pm, *ps;                           // [chunks][R] partial max / sum-exp
    float *ea[kVaeMaxL + 1];                  // encoder outputs [R, e[k+1]] (tanh applied for k < L)
    float *eps, *z;                           // [R, lat/2]
    float *da[kVaeMaxL];                      // decoder hidden outputs [R, d[k+1]] (tanh applied)
    float *LT;                                // logits, item-major [I, R]; dL^T in place during the backward pass
    float *g0, *g1;                           // [R, maxw] gradient ping-pong
};

static int vae_chunks(const VaeDims &v, long long R)
{
    const long long tiles = (R + 31) / 32;
    long long c = ((long long)sm_count() * 4 + tiles - 1) / tiles, cmax = (v.I + 63) / 64;
    if (c > cmax) c = cmax;
    return (int)(c < 1 ? 1 : c);
}

static size_t carve_vae(void *base, const VaeDims &v, int opt, long long R, VaeWs *w, size_t *head = nullptr)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += align256(bytes);
        return p;
    };
    auto f = [&](size_t n) { return (float *)take(sizeof(float) * n); };
    VaeWs t;
    t.hdr = (WsHeader *)take(256);
    t.gN = f((size_t)v.nN);
    t.mN = t.vN = nullptr;
    if (opt == DRB_OPT_ADAM) { t.mN = f((size_t)v.nN); t.vN = f((size_t)v.nN); }
    if (head) *head = off;                    // everything above is zeroed by workspace_init
    const long long chunks = (v.I + 63) / 64;  // upper bound of vae_chunks()
    t.denom = f(R); t.S = f(R); t.lse = f(R);
    t.pm = f((size_t)chunks * R); t.ps = f((size_t)chunks * R);
    for (int k = 0; k <= kVaeMaxL; ++k) t.ea[k] = k < v.ne ? f((size_t)R * v.e[k + 1]) : nullptr;
    t.eps = f((size_t)R * v.half); t.z = f((size_t)R * v.half);
    for (int k = 0; k < kVaeMaxL; ++k) t.da[k] = k < v.L ? f((size_t)R * v.d[k + 1]) : nullptr;
    t.LT = f((size_t)R * v.I);
    t.g0 = f((size_t)R * v.maxw); t.g1 = f((size_t)R * v.maxw);
    if (w) *w = t;
    return off;
}

// ------------------------------------------------------------------------------------------ dropout and eps sources
struct VaeRng {
    const uint32_t *bits;                     // host keep-mask of this step: bit (b * I + i), or nullptr -> Philox
    const float *eps;                         // host eps of this step [B, lat/2], or nullptr -> Philox
    uint32_t k0, k1, ctr, thresh;             // Philox key, per-step counter, keep iff word >= thresh
    float p, scale;                           // dropout rate, 1 / (1 - p)
    int drop;                                 // dropout active (training and p > 0)
};

__device__ __forceinline__ bool vae_keep(const VaeRng &g, long long b, int I, int i)
{
    const unsigned long long e = (unsigned long long)b * (unsigned long long)I + (unsigned long long)i;
    if (g.bits) return (__ldg(g.bits + (e >> 5)) >> (unsigned)(e & 31ull)) & 1u;
    uint32_t c[4] = {(uint32_t)(e >> 2), (uint32_t)(e >> 34), 0x56414531u, g.ctr};
    philox4x32(c, g.k0, g.k1);
    const unsigned q = (unsigned)(e & 3ull);
    return (q == 0 ? c[0] : q == 1 ? c[1] : q == 2 ? c[2] : c[3]) >= g.thresh;
}

// dropped input of the first Linear at nonzero (b, i): F.dropout(F.normalize(R))[b, i]
__device__ __forceinline__ float vae_coef(const VaeRng &g, long long b, int I, int i, float r, float denom)
{
    const float x = r / denom;
    if (!g.drop) return x;
    return vae_keep(g, b, I, i) ? x * g.scale : 0.f;
}

// ------------------------------------------------------------------------------------------ kernels
// one warp per batch row: denom = max(||r||, 1e-12) (F.normalize), S = sum r
__global__ void __launch_bounds__(256) vae_row_stats_kernel(const int64_t *__restrict__ rp, const float *__restrict__ val,
                                                            const int32_t *__restrict__ users, long long B,
                                                            float *__restrict__ denom, float *__restrict__ S)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long b = warp; b < B; b += nw) {
        const int u = users[b];
        double ss = 0.0, s = 0.0;
        for (long long k = rp[u] + lane; k < rp[u + 1]; k += 32) {
            const double r = (double)val[k];
            ss += r * r;
            s += r;
        }
        ss = warp_sum(ss);
        s = warp_sum(s);
        if (lane == 0) {
            const float n = (float)sqrt(ss);
            denom[b] = n > 1e-12f ? n : 1e-12f;
            S[b] = (float)s;
        }
    }
}

// first encoder Linear over the row's nonzeros: h[b, j] = act(b1[j] + sum_nz coef * W1T[i, j]).  One CTA per row; the
// coefficients (dropout bit / Philox word read once per nonzero) are staged in shared memory, threads own columns.
__global__ void __launch_bounds__(256) vae_sparse_enc_kernel(const int64_t *__restrict__ rp, const int32_t *__restrict__ col,
                                                             const float *__restrict__ val, const int32_t *__restrict__ users,
                                                             const float *__restrict__ denom, const float *__restrict__ W1T,
                                                             const float *__restrict__ b1, int I, int H, int act, VaeRng g,
                                                             float *__restrict__ out)
{
    __shared__ float s_c[256];
    __shared__ int s_i[256];
    const long long b = blockIdx.x;
    const int u = users[b];
    const long long k0 = rp[u], k1 = rp[u + 1];
    const float dn = denom[b];
    for (int j0 = 0; j0 < H; j0 += 4 * 256) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (long long t0 = k0; t0 < k1; t0 += 256) {
            __syncthreads();
            const long long k = t0 + threadIdx.x;
            if (k < k1) {
                const int i = col[k];
                s_i[threadIdx.x] = i;
                s_c[threadIdx.x] = vae_coef(g, b, I, i, val[k], dn);
            }
            __syncthreads();
            const int n = (int)(k1 - t0 < 256 ? k1 - t0 : 256);
            for (int q = 0; q < n; ++q) {
                const float c = s_c[q];
                if (c == 0.f) continue;
                const float *w = W1T + (size_t)s_i[q] * H;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int j = j0 + e * 256 + threadIdx.x;
                    if (j < H) acc[e] = fmaf(c, __ldg(w + j), acc[e]);
                }
            }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = j0 + e * 256 + threadIdx.x;
            if (j < H) {
                const float v = b1[j] + acc[e];
                out[b * H + j] = act ? tanhf(v) : v;
            }
        }
    }
}

// gW1T[i, :] += coef * dz[b, :] for every kept nonzero of row b (one CTA per row)
__global__ void __launch_bounds__(256) vae_sparse_wgrad_kernel(const int64_t *__restrict__ rp, const int32_t *__restrict__ col,
                                                               const float *__restrict__ val, const int32_t *__restrict__ users,
                                                               const float *__restrict__ denom, const float *__restrict__ dz,
                                                               int I, int H, VaeRng g, float *__restrict__ gW1T)
{
    __shared__ float s_c[256];
    __shared__ int s_i[256];
    const long long b = blockIdx.x;
    const int u = users[b];
    const long long k0 = rp[u], k1 = rp[u + 1];
    const float dn = denom[b];
    for (long long t0 = k0; t0 < k1; t0 += 256) {
        __syncthreads();
        const long long k = t0 + threadIdx.x;
        if (k < k1) {
            const int i = col[k];
            s_i[threadIdx.x] = i;
            s_c[threadIdx.x] = vae_coef(g, b, I, i, val[k], dn);
        }
        __syncthreads();
        const int n = (int)(k1 - t0 < 256 ? k1 - t0 : 256);
        for (int q = 0; q < n; ++q) {
            const float c = s_c[q];
            if (c == 0.f) continue;
            float *gw = gW1T + (size_t)s_i[q] * H;
            for (int j = threadIdx.x; j < H; j += 256) atomicAdd(gw + j, c * dz[b * H + j]);
        }
    }
}

// z = x + b (Linear bias), then tanh when act: in place on [rows, N]
__global__ void vae_bias_act_kernel(float *__restrict__ x, const float *__restrict__ bias, long long total, int N, int act)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const float v = x[k] + bias[(int)(k % N)];
        x[k] = act ? tanhf(v) : v;
    }
}

// x *= 1 - a^2 (backward of a Tanh whose output is a)
__global__ void vae_tanh_bwd_kernel(float *__restrict__ x, const float *__restrict__ a, long long total)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const float t = a[k];
        x[k] = x[k] * (1.f - t * t);
    }
}

// gb[n] += sum_m dZ[m, n] for any N (one thread per column, rows strided over grid.y)
__global__ void vae_colsum_kernel(const float *__restrict__ dZ, long long M, int N, float *__restrict__ gb)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float s = 0.f;
    for (long long m = blockIdx.y; m < M; m += gridDim.y) s += dZ[m * N + n];
    if (s != 0.f) atomicAdd(gb + n, s);
}

__device__ __forceinline__ float vae_normal(const VaeRng &g, long long e)
{
    // Box-Muller on one Philox block: words 0, 1 -> two uniforms in (0, 1]
    uint32_t c[4] = {(uint32_t)e, (uint32_t)((unsigned long long)e >> 32), 0x56414532u, g.ctr};
    philox4x32(c, g.k0, g.k1);
    const float u1 = ((float)c[0] + 1.f) * 2.3283064e-10f, u2 = (float)c[1] * 2.3283064e-10f;
    return sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
}

// z = eps * exp(0.5 lv) + mu (training) or mu; KL row terms sum(1 + lv - mu^2 - e^lv) into acc (fp64)
__global__ void __launch_bounds__(256) vae_reparam_kernel(const float *__restrict__ h, long long B, int lat, int half, int lvo,
                                                          int training, VaeRng g, float *__restrict__ eps, float *__restrict__ z,
                                                          double *__restrict__ acc)
{
    double kl = 0.0;
    const long long total = B * half;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long b = k / half;
        const int j = (int)(k - b * half);
        const float mu = h[b * lat + j], lv = h[b * lat + lvo + j];
        if (training) {
            const float ep = g.eps ? g.eps[k] : vae_normal(g, k);
            eps[k] = ep;
            z[k] = ep * expf(0.5f * lv) + mu;
        } else {
            z[k] = mu;
        }
        kl += (double)(((1.f + lv) - mu * mu) - expf(lv));
    }
    kl = warp_sum(kl);
    if ((threadIdx.x & 31) == 0 && kl != 0.0) atomicAdd(acc, kl);
}

// d h_enc from d z and the KL term: dmu = dz + c mu, dlv = dz * eps * 0.5 std + 0.5 c (e^lv - 1), c = anneal / B;
// the middle column of an odd latent_dim gets 0
__global__ void vae_reparam_bwd_kernel(const float *__restrict__ h, const float *__restrict__ eps, const float *__restrict__ dz,
                                       long long B, int lat, int half, int lvo, float c, float *__restrict__ dh)
{
    const long long total = B * lat;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const long long b = k / lat;
        const int j = (int)(k - b * lat);
        float v = 0.f;
        if (j < half) {
            v = dz[b * half + j] + c * h[k];
        } else if (j >= lvo) {
            const int q = j - lvo;
            const float lv = h[k], sd = expf(0.5f * lv);
            v = dz[b * half + q] * eps[b * half + q] * 0.5f * sd + 0.5f * c * (expf(lv) - 1.f);
        }
        dh[k] = v;
    }
}

// pass 1 of the softmax over item-major logits LT [I, ld]: CTA (column tile of 32, item chunk) -> online max / sum-exp
// per column over its items.  Lane = column (coalesced), the 8 warps stride over the chunk's items.
__global__ void __launch_bounds__(256) vae_lse_part_kernel(const float *__restrict__ LT, const float *__restrict__ bo, int I,
                                                           long long B, long long ld, int chunk, float *__restrict__ pm,
                                                           float *__restrict__ ps)
{
    __shared__ float s_m[8][32], s_s[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * 32 + lane;
    const int i0 = blockIdx.y * chunk, i1 = min(I, i0 + chunk);
    float m = -INFINITY, s = 0.f;
    if (b < B)
        for (int i = i0 + warp; i < i1; i += 8) {
            const float x = LT[(size_t)i * ld + b] + bo[i];
            if (x > m) { s = s * expf(m - x) + 1.f; m = x; }
            else s += expf(x - m);
        }
    s_m[warp][lane] = m; s_s[warp][lane] = s;
    __syncthreads();
    if (warp == 0 && b < B) {
        float M = -INFINITY;
        for (int q = 0; q < 8; ++q) M = fmaxf(M, s_m[q][lane]);
        float t = 0.f;
        if (M != -INFINITY)
            for (int q = 0; q < 8; ++q) t += s_s[q][lane] * expf(s_m[q][lane] - M);
        pm[(size_t)blockIdx.y * B + b] = M;
        ps[(size_t)blockIdx.y * B + b] = t;
    }
}

// pass 2: combine the chunks -> lse[b]; then one warp per row sums CE_b = sum_nz r (logit - lse) into acc (fp64)
__global__ void __launch_bounds__(256) vae_lse_ce_kernel(const float *__restrict__ pm, const float *__restrict__ ps, int chunks,
                                                         const float *__restrict__ LT, const float *__restrict__ bo,
                                                         long long ld, const int64_t *__restrict__ rp,
                                                         const int32_t *__restrict__ col, const float *__restrict__ val,
                                                         const int32_t *__restrict__ users, long long B, float *__restrict__ lse,
                                                         double *__restrict__ acc)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    double ce = 0.0;
    for (long long b = warp; b < B; b += nw) {
        float M = -INFINITY;
        for (int c = lane; c < chunks; c += 32) M = fmaxf(M, pm[(size_t)c * B + b]);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, off));
        double t = 0.0;
        for (int c = lane; c < chunks; c += 32) t += (double)ps[(size_t)c * B + b] * exp((double)pm[(size_t)c * B + b] - (double)M);
        t = warp_sum(t);
        const float l = M + (float)log(t);
        if (lane == 0) lse[b] = l;
        const int u = users[b];
        for (long long k = rp[u] + lane; k < rp[u + 1]; k += 32) {
            const int i = col[k];
            ce += (double)(val[k] * ((LT[(size_t)i * ld + b] + bo[i]) - l));
        }
    }
    ce = warp_sum(ce);
    if (lane == 0 && ce != 0.0) atomicAdd(acc, ce);
}

// in place: LT[i, b] <- dL = softmax * S_b / B (the dense part of (softmax S_b - R) / B); gbo[i] += sum_b dL[i, b]
__global__ void __launch_bounds__(256) vae_softmax_grad_kernel(float *__restrict__ LT, const float *__restrict__ bo, int I,
                                                               long long B, long long ld, int chunk, const float *__restrict__ lse,
                                                               const float *__restrict__ S, float invB, float *__restrict__ gbo)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * 32 + lane;
    const int i0 = blockIdx.y * chunk, i1 = min(I, i0 + chunk);
    const float l = b < B ? lse[b] : 0.f, sb = b < B ? S[b] : 0.f;
    for (int i = i0 + warp; i < i1; i += 8) {
        float d = 0.f;
        if (b < B) {
            float *p = LT + (size_t)i * ld + b;
            d = expf((*p + bo[i]) - l) * sb * invB;
            *p = d;
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
        if (lane == 0 && d != 0.f) atomicAdd(gbo + i, d);
    }
}

// the sparse part: dL[i, b] -= r / B at every nonzero, and the same on the output-bias gradient
__global__ void __launch_bounds__(256) vae_ce_grad_fix_kernel(float *__restrict__ LT, long long ld, const int64_t *__restrict__ rp,
                                                              const int32_t *__restrict__ col, const float *__restrict__ val,
                                                              const int32_t *__restrict__ users, long long B, float invB,
                                                              float *__restrict__ gbo)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long b = warp; b < B; b += nw) {
        const int u = users[b];
        for (long long k = rp[u] + lane; k < rp[u + 1]; k += 32) {
            const int i = col[k];
            const float r = val[k] * invB;
            LT[(size_t)i * ld + b] -= r;
            atomicAdd(gbo + i, -r);
        }
    }
}

// loss = CE + KL in the reference's fp32 order; NaN -> sticky status (an infinite loss trains on, as fit() checks isnan only)
__global__ void vae_finalize_kernel(WsHeader *hdr, long long B, float anneal, double *__restrict__ loss_out, long long step)
{
    const double *a = hdr->acc[0];
    const float ce = -(float)(a[0] / (double)B);
    const float kl = (-0.5f * (float)(a[1] / (double)B)) * anneal;
    const float loss = ce + kl;
    *loss_out = (double)loss;
    if (isnan(loss)) { hdr->status = DRB_ERR_NAN_LOSS; hdr->nan_step = step; }
}

// out[r, i] = LT[i, r] + bo[i]   (eval-mode decoder rows, user-major)
__global__ void vae_rows_out_kernel(const float *__restrict__ LT, const float *__restrict__ bo, int I, long long rows,
                                    float *__restrict__ out)
{
    __shared__ float t[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;             // 256 threads: 32 x 8
    const long long r0 = (long long)blockIdx.y * 32;
    const int i0 = blockIdx.x * 32;
    for (int q = ty; q < 32; q += 8) {
        const int i = i0 + q;
        const long long r = r0 + tx;
        t[q][tx] = (i < I && r < rows) ? LT[(size_t)i * rows + r] + bo[i] : 0.f;
    }
    __syncthreads();
    for (int q = ty; q < 32; q += 8) {
        const long long r = r0 + q;
        const int i = i0 + tx;
        if (r < rows && i < I) out[(size_t)r * I + i] = t[tx][q];
    }
}

// candidate scores: one warp per (row, candidate): <hidden[row], W_out[c]> + b_out[c]
__global__ void __launch_bounds__(256) vae_cand_score_kernel(const float *__restrict__ hid, int K, const float *__restrict__ Wo,
                                                             const float *__restrict__ bo, const int64_t *__restrict__ cands,
                                                             long long n, int C, float *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long q = warp; q < n * C; q += nw) {
        const long long r = q / C;
        const long long c = cands[q];
        float s = 0.f;
        for (int k = lane; k < K; k += 32) s = fmaf(hid[r * K + k], __ldg(Wo + (size_t)c * K + k), s);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane == 0) out[q] = s + bo[c];
    }
}

// ------------------------------------------------------------------------------------------ host sequencing
struct VaeCsr {
    const int64_t *rp;
    const int32_t *col;
    const float *val;
};

static int vae_bias_act(float *x, const float *b, long long rows, int N, int act, cudaStream_t st)
{
    vae_bias_act_kernel<<<grid_size(rows * N, 256), 256, 0, st>>>(x, b, rows * N, N, act);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

static int vae_colsum(const float *dZ, long long M, int N, float *gb, cudaStream_t st)
{
    long long gy = (long long)sm_count() * 8 / ((N + 255) / 256);
    if (gy > M) gy = M;
    if (gy < 1) gy = 1;
    vae_colsum_kernel<<<dim3((unsigned)((N + 255) / 256), (unsigned)gy), 256, 0, st>>>(dZ, M, N, gb);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

// encoder + reparameterisation + decoder hidden layers on B rows; leaves the last decoder hidden in w.da[L-1] (or w.z)
static int vae_forward_hidden(const VaeDims &v, const VaeWs &w, const float *N, const VaeCsr &R, const int32_t *users, long long B,
                              int training, const VaeRng &g, int dtype, cudaStream_t st)
{
    vae_row_stats_kernel<<<grid_size(B * 32, 256), 256, 0, st>>>(R.rp, R.val, users, B, w.denom, w.S);
    vae_sparse_enc_kernel<<<(unsigned)B, 256, 0, st>>>(R.rp, R.col, R.val, users, w.denom, N + v.oEW[0], N + v.oEB[0], v.I, v.e[1],
                                                       v.L > 0 ? 1 : 0, g, w.ea[0]);
    DRB_CUDA(cudaGetLastError());
    for (int k = 1; k < v.ne; ++k) {
        int rc = gemm_nt(dtype, B, v.e[k + 1], v.e[k], w.ea[k - 1], v.e[k], N + v.oEW[k], v.e[k], w.ea[k], v.e[k + 1], st);
        if (rc == DRB_OK) rc = vae_bias_act(w.ea[k], N + v.oEB[k], B, v.e[k + 1], k < v.L ? 1 : 0, st);
        if (rc != DRB_OK) return rc;
    }
    vae_reparam_kernel<<<grid_size(B * v.half, 256), 256, 0, st>>>(w.ea[v.L], B, v.lat, v.half, v.lvo, training, g, w.eps, w.z,
                                                                   &w.hdr->acc[0][1]);
    DRB_CUDA(cudaGetLastError());
    const float *x = w.z;
    for (int k = 0; k < v.L; ++k) {
        int rc = gemm_nt(dtype, B, v.d[k + 1], v.d[k], x, v.d[k], N + v.oDW[k], v.d[k], w.da[k], v.d[k + 1], st);
        if (rc == DRB_OK) rc = vae_bias_act(w.da[k], N + v.oDB[k], B, v.d[k + 1], 1, st);
        if (rc != DRB_OK) return rc;
        x = w.da[k];
    }
    return DRB_OK;
}

static const float *vae_last_hidden(const VaeDims &v, const VaeWs &w) { return v.L > 0 ? w.da[v.L - 1] : w.z; }

// LT [I, B] = W_out [I, K] x hidden[B, K]^T, B sliced into panels of <= kVaePanel columns (item dimension = M)
static int vae_logits(const VaeDims &v, const VaeWs &w, const float *N, long long B, int dtype, cudaStream_t st)
{
    const int K = v.d[v.L];
    const float *x = vae_last_hidden(v, w);
    for (long long c0 = 0; c0 < B; c0 += kVaePanel) {
        const int nb = (int)(B - c0 < kVaePanel ? B - c0 : kVaePanel);
        int rc = gemm_nt(dtype, v.I, nb, K, N + v.oDW[v.L], K, x + c0 * K, K, w.LT + c0, B, st);
        if (rc != DRB_OK) return rc;
    }
    return DRB_OK;
}

// one dense Linear backward: dz [B, out] (already through the activation) -> gW [out, in] += dz^T x, gb += colsum dz,
// dx [B, in] = dz W (skipped when dx == nullptr)
static int vae_linear_bwd(int dtype, long long B, int in, int out, const float *x, const float *W, const float *dz, float *gW,
                          float *gb, float *dx, cudaStream_t st)
{
    int rc = vae_colsum(dz, B, out, gb, st);
    if (rc == DRB_OK) rc = gemm_tn_acc_t(dtype, in, out, (int)B, x, in, dz, out, gW, in, st);
    if (rc == DRB_OK && dx) rc = gemm_nn(dtype, B, in, out, dz, out, W, in, dx, in, st);
    return rc;
}

}  // namespace drb

using namespace drb;

extern "C" int64_t drb_vae_param_count(int32_t I, const int32_t *hidden, int32_t L, int32_t lat)
{
    VaeDims v;
    if (!vae_dims(v, I, hidden, L, lat)) return -1;
    return v.nN;
}

extern "C" size_t drb_vae_workspace_bytes(int32_t I, const int32_t *hidden, int32_t L, int32_t lat, int32_t opt, int64_t max_rows)
{
    VaeDims v;
    if (!vae_dims(v, I, hidden, L, lat) || max_rows < 1) return 0;
    return carve_vae(nullptr, v, opt, max_rows, nullptr);
}

extern "C" int drb_vae_workspace_init(void *d_ws, int32_t I, const int32_t *hidden, int32_t L, int32_t lat, int32_t opt,
                                      int64_t max_rows, void *stream)
{
    VaeDims v;
    DRB_REQUIRE(d_ws && vae_dims(v, I, hidden, L, lat) && max_rows >= 1, "vae_workspace_init: bad arguments");
    size_t head = 0;
    carve_vae(nullptr, v, opt, max_rows, nullptr, &head);
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, head, (cudaStream_t)stream));
    return DRB_OK;
}

// n_steps VAECF steps (apply != 0: calc_loss + backward + optimizer.step) or the loss of one batch (apply == 0).
// Step s takes users d_users[(first_step + s) * batch, ...) (a ragged last batch holds the rest).  Its update number is
// update0 + s + 1 (anneal = min(cap, update / total_anneal_steps), or cap when total_anneal_steps <= 0).
// training != 0: dropout p on the normalised input and z = eps * std + mu; keep bits from d_keep (torch's keep-mask of the
// step, [B, item_num] row-major, bit-packed little-endian into 32-bit words, ceil(batch * item_num / 32) words per step) or,
// when NULL, from Philox4x32-10(seed); eps from d_eps ([n_steps][batch][lat/2] fp32) or, when NULL, from Philox + Box-Muller.
extern "C" int drb_vae_train_steps(float *d_N, void *d_ws, int32_t I, const int32_t *hidden, int32_t L, int32_t lat, int64_t max_rows,
                                   const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val, int32_t U,
                                   const int32_t *d_users, int64_t n, int64_t batch, int64_t first_step, int64_t n_steps,
                                   const drb_hyper *h, int64_t adam_step0, int32_t apply, int32_t training, int32_t tower_dtype,
                                   float dropout, const uint32_t *d_keep, const float *d_eps, uint64_t seed, double anneal_cap,
                                   int64_t total_anneal_steps, int64_t update0, double *d_step_loss, int32_t sync_and_check,
                                   int64_t *nan_step, void *stream)
{
    VaeDims v;
    DRB_REQUIRE(d_N && d_ws && d_row_ptr && d_col && d_val && d_users && h && d_step_loss && U > 0, "vae_train_steps: null argument");
    DRB_REQUIRE(vae_dims(v, I, hidden, L, lat), "vae_train_steps: bad dims (item_num > 0, <= 8 hidden layers, latent_dim >= 2)");
    DRB_REQUIRE(batch > 0 && batch <= max_rows, "vae: batch %lld exceeds max_rows=%lld", (long long)batch, (long long)max_rows);
    DRB_REQUIRE(n_steps == 0 || (first_step + n_steps - 1) * batch < n, "vae: steps exceed %lld users", (long long)n);
    DRB_REQUIRE(dropout >= 0.f && dropout < 1.f, "vae: dropout must be in [0, 1)");
    DRB_REQUIRE(h->opt == DRB_OPT_SGD || h->opt == DRB_OPT_ADAM, "vae: SGD and Adam only (optimizer id %d)", h->opt);
    DRB_REQUIRE(tower_dtype == 0 || tower_dtype == 1, "vae: tower_dtype must be 0 (fp32) or 1 (bf16)");
    if (n_steps == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    VaeWs w;
    carve_vae(d_ws, v, h->opt, max_rows, &w);
    const VaeCsr R{d_row_ptr, d_col, d_val};
    const long long mask_words = (batch * (long long)I + 31) / 32;
    const int dt = tower_dtype;
    DRB_CUDA(cudaMemsetAsync(w.hdr, 0, sizeof(WsHeader), st));
    for (int64_t s = 0; s < n_steps; ++s) {
        const int64_t base = (first_step + s) * batch, B = (n - base < batch) ? n - base : batch;
        const int32_t *users = d_users + base;
        const long long upd = update0 + s + 1;
        const double an = total_anneal_steps > 0 ? fmin(anneal_cap, (double)upd / (double)total_anneal_steps) : anneal_cap;
        VaeRng g;
        g.drop = training && dropout > 0.f;
        g.p = dropout;
        g.scale = 1.f / (1.f - dropout);
        g.bits = g.drop && d_keep ? d_keep + (size_t)s * mask_words : nullptr;
        g.eps = training && d_eps ? d_eps + (size_t)s * batch * v.half : nullptr;
        g.k0 = (uint32_t)seed; g.k1 = (uint32_t)(seed >> 32);
        g.ctr = (uint32_t)upd;
        g.thresh = (uint32_t)fmin(4294967295.0, (double)dropout * 4294967296.0);
        DRB_CUDA(cudaMemsetAsync(w.hdr, 0, kHdrResetBytes, st));
        // ---- forward + loss
        int rc = vae_forward_hidden(v, w, d_N, R, users, B, training, g, dt, st);
        if (rc == DRB_OK) rc = vae_logits(v, w, d_N, B, dt, st);
        if (rc != DRB_OK) return rc;
        const float *bo = d_N + v.oDB[v.L];
        const int chunks = vae_chunks(v, B), chunk = (v.I + chunks - 1) / chunks;
        const dim3 sgrid((unsigned)((B + 31) / 32), (unsigned)chunks);
        vae_lse_part_kernel<<<sgrid, 256, 0, st>>>(w.LT, bo, v.I, B, B, chunk, w.pm, w.ps);
        vae_lse_ce_kernel<<<grid_size(B * 32, 256), 256, 0, st>>>(w.pm, w.ps, chunks, w.LT, bo, B, R.rp, R.col, R.val, users, B, w.lse,
                                                                  &w.hdr->acc[0][0]);
        vae_finalize_kernel<<<1, 1, 0, st>>>(w.hdr, B, (float)an, d_step_loss + s, first_step + s);
        DRB_CUDA(cudaGetLastError());
        if (!apply) break;
        // ---- backward: output layer (item-major dL^T)
        const float invB = 1.f / (float)B;
        vae_softmax_grad_kernel<<<sgrid, 256, 0, st>>>(w.LT, bo, v.I, B, B, chunk, w.lse, w.S, invB, w.gN + v.oDB[v.L]);
        vae_ce_grad_fix_kernel<<<grid_size(B * 32, 256), 256, 0, st>>>(w.LT, B, R.rp, R.col, R.val, users, B, invB, w.gN + v.oDB[v.L]);
        DRB_CUDA(cudaGetLastError());
        const int K = v.d[v.L];
        const float *xl = vae_last_hidden(v, w);
        for (int c0 = 0; c0 < K; c0 += kVaePanel) {                       // gW_out [I, K] = dL^T x hidden   (M = I)
            const int nk = K - c0 < kVaePanel ? K - c0 : kVaePanel;
            rc = gemm_nn(dt, v.I, nk, (int)B, w.LT, B, xl + c0, K, w.gN + v.oDW[v.L] + c0, K, st);
            if (rc != DRB_OK) return rc;
        }
        DRB_CUDA(cudaMemsetAsync(w.g0, 0, sizeof(float) * (size_t)B * K, st));
        for (long long c0 = 0; c0 < B; c0 += kVaePanel) {                 // d hidden [B, K] += (W_out^T dL^T)^T   (split-K over I)
            const int nb = (int)(B - c0 < kVaePanel ? B - c0 : kVaePanel);
            rc = gemm_tn_acc_t(dt, K, nb, v.I, d_N + v.oDW[v.L], K, w.LT + c0, B, w.g0 + c0 * K, K, st);
            if (rc != DRB_OK) return rc;
        }
        // ---- decoder hidden layers
        float *gcur = w.g0, *gnext = w.g1;
        for (int k = v.L - 1; k >= 0; --k) {
            vae_tanh_bwd_kernel<<<grid_size(B * v.d[k + 1], 256), 256, 0, st>>>(gcur, w.da[k], B * v.d[k + 1]);
            DRB_CUDA(cudaGetLastError());
            const float *x = k > 0 ? w.da[k - 1] : w.z;
            rc = vae_linear_bwd(dt, B, v.d[k], v.d[k + 1], x, d_N + v.oDW[k], gcur, w.gN + v.oDW[k], w.gN + v.oDB[k], gnext, st);
            if (rc != DRB_OK) return rc;
            float *t = gcur; gcur = gnext; gnext = t;
        }
        // ---- reparameterisation + KL -> d h_enc [B, lat]
        const float c = (float)an * invB;
        vae_reparam_bwd_kernel<<<grid_size(B * v.lat, 256), 256, 0, st>>>(w.ea[v.L], w.eps, gcur, B, v.lat, v.half, v.lvo, c, gnext);
        DRB_CUDA(cudaGetLastError());
        { float *t = gcur; gcur = gnext; gnext = t; }
        // ---- encoder dense layers (k >= 1), then the sparse first layer
        for (int k = v.L; k >= 1; --k) {
            if (k < v.L) {
                vae_tanh_bwd_kernel<<<grid_size(B * v.e[k + 1], 256), 256, 0, st>>>(gcur, w.ea[k], B * v.e[k + 1]);
                DRB_CUDA(cudaGetLastError());
            }
            rc = vae_linear_bwd(dt, B, v.e[k], v.e[k + 1], w.ea[k - 1], d_N + v.oEW[k], gcur, w.gN + v.oEW[k], w.gN + v.oEB[k], gnext, st);
            if (rc != DRB_OK) return rc;
            float *t = gcur; gcur = gnext; gnext = t;
        }
        if (v.L > 0) {
            vae_tanh_bwd_kernel<<<grid_size(B * v.e[1], 256), 256, 0, st>>>(gcur, w.ea[0], B * v.e[1]);
            DRB_CUDA(cudaGetLastError());
        }
        rc = vae_colsum(gcur, B, v.e[1], w.gN + v.oEB[0], st);
        if (rc != DRB_OK) return rc;
        vae_sparse_wgrad_kernel<<<(unsigned)B, 256, 0, st>>>(R.rp, R.col, R.val, users, w.denom, gcur, v.I, v.e[1], g, w.gN + v.oEW[0]);
        DRB_CUDA(cudaGetLastError());
        // ---- update
        rc = dense_update(d_N, w.gN, w.mN, w.vN, v.nN, h, adam_step0 + s, w.hdr, st);
        if (rc != DRB_OK) return rc;
    }
    if (sync_and_check) return check_nan(d_ws, st, nan_step);
    return DRB_OK;
}

// eval-mode forward (no dropout, z = mu) for users d_users[0, n): what = 0 -> decoder output rows [n, item_num];
// 1 -> last decoder hidden rows [n, d_L] (drb_vae_candidate_scores' input); 2 -> encoder output rows [n, latent_dim]
extern "C" int drb_vae_forward(const float *d_N, void *d_ws, int32_t I, const int32_t *hidden, int32_t L, int32_t lat, int32_t opt,
                               int64_t max_rows, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val, int32_t U,
                               const int32_t *d_users, int64_t n, int32_t what, int32_t tower_dtype, float *d_out, void *stream)
{
    VaeDims v;
    DRB_REQUIRE(d_N && d_ws && d_row_ptr && d_col && d_val && d_users && d_out && n >= 0 && U > 0, "vae_forward: null argument");
    DRB_REQUIRE(vae_dims(v, I, hidden, L, lat) && max_rows >= 1 && what >= 0 && what <= 2, "vae_forward: bad arguments");
    DRB_REQUIRE(tower_dtype == 0 || tower_dtype == 1, "vae: tower_dtype must be 0 (fp32) or 1 (bf16)");
    cudaStream_t st = (cudaStream_t)stream;
    VaeWs w;
    carve_vae(d_ws, v, opt, max_rows, &w);
    const VaeCsr R{d_row_ptr, d_col, d_val};
    VaeRng g{};
    const int K = v.d[v.L];
    for (long long r0 = 0; r0 < n; r0 += max_rows) {
        const long long rows = n - r0 < max_rows ? n - r0 : max_rows;
        int rc = vae_forward_hidden(v, w, d_N, R, d_users + r0, rows, 0, g, tower_dtype, st);
        if (rc != DRB_OK) return rc;
        if (what == 2) {
            DRB_CUDA(cudaMemcpyAsync(d_out + r0 * v.lat, w.ea[v.L], sizeof(float) * rows * v.lat, cudaMemcpyDeviceToDevice, st));
        } else if (what == 1) {
            DRB_CUDA(cudaMemcpyAsync(d_out + r0 * K, vae_last_hidden(v, w), sizeof(float) * rows * K, cudaMemcpyDeviceToDevice, st));
        } else {
            rc = vae_logits(v, w, d_N, rows, tower_dtype, st);
            if (rc != DRB_OK) return rc;
            dim3 grid((unsigned)((v.I + 31) / 32), (unsigned)((rows + 31) / 32));
            vae_rows_out_kernel<<<grid, 256, 0, st>>>(w.LT, d_N + v.oDB[v.L], v.I, rows, d_out + r0 * v.I);
            DRB_CUDA(cudaGetLastError());
        }
    }
    return DRB_OK;
}

// scores[r, c] = <d_hidden[r], W_out[cands[r, c]]> + b_out[cands[r, c]]: the decoder output at the candidates only
extern "C" int drb_vae_candidate_scores(const float *d_N, int32_t I, const int32_t *hidden, int32_t L, int32_t lat,
                                        const float *d_hidden, int64_t n, const int64_t *d_cands, int32_t C, float *d_scores,
                                        void *stream)
{
    VaeDims v;
    DRB_REQUIRE(d_N && d_hidden && d_cands && d_scores && n >= 0 && C > 0, "vae_candidate_scores: null argument");
    DRB_REQUIRE(vae_dims(v, I, hidden, L, lat), "vae_candidate_scores: bad dims");
    if (n == 0) return DRB_OK;
    const int K = v.d[v.L];
    vae_cand_score_kernel<<<grid_size(n * C * 32, 256), 256, 0, (cudaStream_t)stream>>>(d_hidden, K, d_N + v.oDW[v.L], d_N + v.oDB[v.L],
                                                                                       d_cands, n, C, d_scores);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}
