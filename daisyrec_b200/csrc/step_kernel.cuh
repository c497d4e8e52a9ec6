// step_kernel.cuh -- device code of the BPR step kernel (see the header of mf_bpr.cu for the algorithm), shared by the
// single-GPU persistent kernel (mf_bpr.cu) and the peer-exchange multi-GPU kernel (p2p.cu).  The body is a template over an
// EXCHANGE policy: NoExchange compiles to exactly the single-GPU kernel; P2PExchange (p2p.cu) redirects the item-side
// accumulators into a peer-visible buffer, rendezvouses with the other ranks between the phases and replaces the item half of
// the phase-2 sweep with a reduce-update-broadcast of this rank's item slice over NVLink.
#pragma once
#include <math.h>
#include <stdlib.h>

#include "step.cuh"

namespace drb {

constexpr int kThreads = 256;
constexpr int kTileMax = 1024;  // triples per staged index tile

constexpr int kTileDefault = 512;

// Tile size for `per_cta` triples per CTA and step: the fewest equal tiles of at most `cap` triples (a multiple of 16), so every
// CTA walks the same number of full tiles (cap 512: 3 543 per CTA -> 7 tiles of 512; cap 1 024 -> 4 tiles of 896).
inline int pick_tile(long long per_cta, int cap = kTileDefault)
{
    static const int forced = [] {
        const char *e = getenv("DRB_TILE_CAP");   // developer switch
        int c = e ? atoi(e) : 0;
        return (c >= 16 && c <= kTileMax) ? c / 16 * 16 : 0;
    }();
    if (forced) cap = forced;
    if (cap > kTileMax) cap = kTileMax;
    if (cap < 16) cap = 16;
    if (per_cta < 16) return 16;
    const long long k = (per_cta + cap - 1) / cap;
    long long tile = ((per_cta + k - 1) / k + 15) / 16 * 16;
    return (int)(tile > cap ? cap : tile);
}
#ifndef DRB_MINB
#define DRB_MINB 2             // resident CTAs per SM the register allocator must allow
#endif
#ifndef DRB_UNR
#define DRB_UNR 2              // triples in flight per lane group (memory-level parallelism)
#endif

// ------------------------------------------------------------------ device pieces
__device__ __forceinline__ float sgnf(float x) { return (float)((x > 0.f) - (x < 0.f)); }

struct Norms {
    float inv_u, inv_i, inv_j;  // 1/||.||_F, 0 when the norm is 0 (zero subgradient)
};

struct AdamCoef {
    float step_size, bc2_sqrt;
};

// Apply the accumulated gradient of ONE table row (all W lanes of the group cooperate).
// cnt_a / cnt_b: occurrences weighted by inv_a / inv_b (user rows: cnt_b = 0).
template <int VEC, int W, int NCH, int OPT>
__device__ __forceinline__ void apply_row(float *theta_row, float *g_row, float *m_row, float *v_row, int gl,
                                          int chunks, float cnt_a, float inv_a, float cnt_b, float inv_b,
                                          const StepParams &p, const AdamCoef &ac, bool touched)
{
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        int c = gl + ch * W;
        if (c >= chunks) continue;
        float *tp = theta_row + c * VEC;
        Vec<VEC> th = ld_row<VEC>(tp);
        Vec<VEC> g;
        if (touched) {
            g = ld_row<VEC>(g_row + c * VEC);
            Vec<VEC> z;
#pragma unroll
            for (int e = 0; e < VEC; ++e) z.v[e] = 0.f;
            st_row<VEC>(g_row + c * VEC, z);
        } else {
#pragma unroll
            for (int e = 0; e < VEC; ++e) g.v[e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            float t = th.v[e];
            float gg = g.v[e];
            if (touched) {
                float sg = p.reg1 * sgnf(t);
                gg += cnt_a * (sg + p.reg2 * t * inv_a) + cnt_b * (sg + p.reg2 * t * inv_b);
            }
            g.v[e] = gg;
        }
        if constexpr (OPT == DRB_OPT_SGD) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) th.v[e] = th.v[e] - p.lr * g.v[e];
        } else {
            Vec<VEC> m = ld_row<VEC>(m_row + c * VEC), v = ld_row<VEC>(v_row + c * VEC);
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                float gk = g.v[e];
                m.v[e] = m.v[e] + (gk - m.v[e]) * (1.f - p.beta1);
                v.v[e] = v.v[e] * p.beta2 + (1.f - p.beta2) * gk * gk;
                float denom = sqrtf(v.v[e]) / ac.bc2_sqrt + p.eps;
                th.v[e] = th.v[e] - ac.step_size * (m.v[e] / denom);
            }
            st_row<VEC>(m_row + c * VEC, m);
            st_row<VEC>(v_row + c * VEC, v);
        }
        st_row<VEC>(tp, th);
    }
}

// Dense phase-2 sweep: lane groups walk ALL rows of P then Q, R rows in flight each.  Counter, theta
// and gradient accumulator of the R rows are loaded unconditionally and up front (one memory round
// trip instead of three dependent ones); an untouched SGD row has cnt == 0 and g == 0, so nothing is
// written for it.  Adam moves every row (dense optimiser semantics of the reference).  Adagrad / RMSprop
// (AbstractRecommender.py:57-60, torch defaults) keep ONE state row in the m slot: Adagrad leaves an untouched row
// alone (g = 0 adds nothing), RMSprop's running square of an untouched row still decays by alpha.
template <int VEC, int W, int NCH, int OPT, bool USERS_ONLY = false>
__device__ __forceinline__ void dense_sweep(const StepParams &p, const Norms &nm, const AdamCoef &ac, int gl, int group,
                                            int groups_per_cta, int chunks)
{
    constexpr int R = (OPT == DRB_OPT_SGD) ? ((NCH * VEC <= 4) ? 4 : 2) : ((NCH * VEC <= 4) ? 2 : 1);
    const long long rows = USERS_ONLY ? (long long)p.U : (long long)p.U + p.I;   // peer exchange: item rows have an owner rank
    const long long tg = (long long)gridDim.x * groups_per_cta;
    const int F = p.F;
    for (long long r0 = (long long)blockIdx.x * groups_per_cta + group; r0 < rows; r0 += tg * R) {
        float *th_p[R], *g_p[R], *m_p[R], *v_p[R];
        unsigned long long cnt[R];
        bool act[R], is_user[R];
        Row<VEC, W, NCH> th[R], g[R], m[R], v[R];
#pragma unroll
        for (int k = 0; k < R; ++k) {
            long long r = r0 + (long long)k * tg;
            act[k] = r < rows;
            is_user[k] = r < p.U;
            long long it = is_user[k] ? r : r - p.U;
            size_t o = (size_t)(act[k] ? it : 0) * F;
            th_p[k] = (is_user[k] ? p.P : p.Q) + o;
            g_p[k] = (is_user[k] ? p.ws.gP : p.ws.gQ) + o;
            cnt[k] = 0;
            if (act[k]) cnt[k] = is_user[k] ? (unsigned long long)__ldcg(p.ws.cntU + it) : __ldcg(p.ws.cntI + it);
            th[k] = load_row<VEC, W, NCH>(th_p[k], gl, chunks, act[k]);
            g[k] = load_row<VEC, W, NCH>(g_p[k], gl, chunks, act[k]);
            if constexpr (OPT != DRB_OPT_SGD) {
                m_p[k] = (is_user[k] ? p.ws.mP : p.ws.mQ) + o;
                m[k] = load_row<VEC, W, NCH>(m_p[k], gl, chunks, act[k]);
            }
            if constexpr (OPT == DRB_OPT_ADAM) {
                v_p[k] = (is_user[k] ? p.ws.vP : p.ws.vQ) + o;
                v[k] = load_row<VEC, W, NCH>(v_p[k], gl, chunks, act[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < R; ++k) {
            const bool touched = cnt[k] != 0;
            if (!act[k] || ((OPT == DRB_OPT_SGD || OPT == DRB_OPT_ADAGRAD) && !touched && !p.dense_grad)) continue;
            const float ca = (float)(unsigned)(cnt[k] & 0xffffffffull), cb = p.neg_mult * (float)(unsigned)(cnt[k] >> 32);
            const float ia = is_user[k] ? nm.inv_u : nm.inv_i, ib = nm.inv_j;
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                int c = gl + ch * W;
                if (c >= chunks) continue;
                Vec<VEC> &t = th[k].c[ch];
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    float x = t.v[e], gg = p.gscale * g[k].c[ch].v[e];
                    if (touched) {
                        float sg = p.reg1 * sgnf(x);
                        gg += ca * (sg + p.reg2 * x * ia) + cb * (sg + p.reg2 * x * ib);
                    }
                    if constexpr (OPT == DRB_OPT_SGD) {
                        t.v[e] = x - p.lr * gg;
                    } else if constexpr (OPT == DRB_OPT_ADAGRAD) {   // sum += g^2; theta -= lr g / (sqrt(sum) + 1e-10)
                        float ss = m[k].c[ch].v[e] + gg * gg;
                        t.v[e] = x - p.lr * (gg / (sqrtf(ss) + 1e-10f));
                        m[k].c[ch].v[e] = ss;
                    } else if constexpr (OPT == DRB_OPT_RMSPROP) {   // sq = .99 sq + .01 g^2; theta -= lr g / (sqrt(sq) + 1e-8)
                        float sq = m[k].c[ch].v[e] * 0.99f + (1.f - 0.99f) * gg * gg;
                        t.v[e] = x - p.lr * (gg / (sqrtf(sq) + 1e-8f));
                        m[k].c[ch].v[e] = sq;
                    } else {
                        float mm = m[k].c[ch].v[e], vv = v[k].c[ch].v[e];
                        mm = mm + (gg - mm) * (1.f - p.beta1);
                        vv = vv * p.beta2 + (1.f - p.beta2) * gg * gg;
                        float denom = sqrtf(vv) / ac.bc2_sqrt + p.eps;
                        t.v[e] = x - ac.step_size * (mm / denom);
                        m[k].c[ch].v[e] = mm;
                        v[k].c[ch].v[e] = vv;
                    }
                }
                st_row<VEC>(th_p[k] + c * VEC, t);
                if constexpr (OPT != DRB_OPT_SGD) st_row<VEC>(m_p[k] + c * VEC, m[k].c[ch]);
                if constexpr (OPT == DRB_OPT_ADAM) st_row<VEC>(v_p[k] + c * VEC, v[k].c[ch]);
                if (touched) {
                    Vec<VEC> z;
#pragma unroll
                    for (int e = 0; e < VEC; ++e) z.v[e] = 0.f;
                    st_row<VEC>(g_p[k] + c * VEC, z);
                }
            }
            if (touched && gl == 0 && !p.keep_counts) {
                long long r = r0 + (long long)k * tg;
                if (is_user[k]) p.ws.cntU[r] = 0u; else p.ws.cntI[r - p.U] = 0ull;
            }
        }
    }
}

// Fresh uniform negative for (user u, global triple index gt, step): a Philox word scaled to [0, n_comp) by multiply-high,
// then the k-th item missing from the user's sorted row: item = k + #{s : col[s] - s <= k} (one binary search).
__device__ __forceinline__ int draw_negative(const StepParams &p, int u, unsigned long long gt, unsigned long long step)
{
    const long long rb = p.neg_row_ptr[u], re = p.neg_row_ptr[u + 1];
    const unsigned n_comp = (unsigned)((long long)p.I - (re - rb));
    uint32_t c[4] = {(uint32_t)gt, (uint32_t)(gt >> 32), (uint32_t)step, (uint32_t)(step >> 32)};
    philox4x32(c, (uint32_t)p.neg_seed, (uint32_t)(p.neg_seed >> 32));
    const int k = (int)__umulhi(c[0], n_comp);
    long long lo = 0, hi = re - rb;
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if ((long long)__ldg(p.neg_col + rb + mid) - mid <= (long long)k) lo = mid + 1; else hi = mid;
    }
    const int item = k + (int)lo;
    return item < p.I ? item : p.I - 1;   // only reachable for a user who interacted with every item (rejected by the host)
}

template <bool LEAN> struct RowOffset { typedef size_t type; };
template <> struct RowOffset<true> { typedef unsigned type; };

// deterministic mode: contribution -> 2^40 fixed point (|sum| < 8.3e6, resolution 9e-13), scalars -> 2^24
constexpr double kDetScale = 1099511627776.0, kDetAccScale = 16777216.0;
__device__ __forceinline__ void det_red(long long *p, float v)
{
    red_add_u64(reinterpret_cast<unsigned long long *>(p), (unsigned long long)__double2ll_rn((double)v * kDetScale));
}

// Exchange policy of the single-GPU kernel: nothing to exchange (every hook is a compile-time no-op).
struct NoExchange {
    static constexpr bool kActive = false;
    __device__ __forceinline__ void begin_step(StepParams &, long long, double *&) {}
    __device__ __forceinline__ bool after_phase1(const StepParams &, long long, double *&, unsigned long long &) { return true; }
    template <int VEC, int W, int NCH>
    __device__ __forceinline__ void item_slice(const StepParams &, long long, const Norms &, const AdamCoef &, int, int, int,
                                               int, unsigned long long &) {}
    __device__ __forceinline__ bool end_step(const StepParams &, long long, unsigned long long &) { return true; }
};

// LEAN: the MF hot instantiation (launch_steps picks it when the parameters allow): BPR, no ego / norm tables (LightGCN),
// no in-kernel negative draw, and 32-bit element offsets into the tables (rows * F < 2^32) -- the same arithmetic on the same
// operands in the same order as the general body, with ~1/3 fewer instructions per triple.
template <int VEC, int W, int NCH, bool GEN, class XCH, bool LEAN = false>
__device__ __forceinline__ void bpr_steps_body(StepParams &p, XCH &xch)
{
    static_assert(!(GEN && LEAN), "the lean body is BPR only");
    using RowOff = typename RowOffset<LEAN>::type;
    constexpr int GPW = 32 / W;                  // lane groups per warp
    constexpr int GROUPS = (kThreads / 32) * GPW;  // lane groups per CTA
    constexpr int UNR = (NCH * VEC <= (LEAN ? 8 : 4)) ? DRB_UNR : 1;  // triples in flight per group

    __shared__ __align__(128) int32_t s_idx[2][3][kTileMax];
    __shared__ uint64_t s_bar[2];
    __shared__ double s_red[8][kThreads / 32];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gl = lane % W, gw = lane / W;
    const int group = warp * GPW + gw;
    const int chunks = p.F / VEC;
    const int F = p.F;
    WsHeader *hdr = p.ws.hdr;

    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (*(volatile int *)&hdr->status != 0) return;   // split mode: a previous step already raised NaN
    uint32_t par0 = 0, par1 = 0;
    unsigned long long epoch = 0;
    const int tile = p.tile;
    const bool pw = GEN && p.loss >= DRB_LOSS_CL;   // point-wise: bj is the label plane, no negative row

    // stage one index tile: TMA bulk copy when full and 16-byte aligned, plain loads otherwise
    auto stage = [&](long long tbase, int cnt, int b) {
        const int32_t *su = p.bu + tbase, *si = p.bi + tbase, *sj = p.bj + tbase;
        bool bulk = (cnt % 4 == 0) && ((((uintptr_t)su | (uintptr_t)si | (uintptr_t)sj) & 15) == 0);
        if (bulk) {
            if (tid == 0) {
                uint32_t bytes = (uint32_t)cnt * 4u;
                mbar_expect_tx(&s_bar[b], 3u * bytes);
                tma_load_1d(&s_idx[b][0][0], su, bytes, &s_bar[b]);
                tma_load_1d(&s_idx[b][1][0], si, bytes, &s_bar[b]);
                tma_load_1d(&s_idx[b][2][0], sj, bytes, &s_bar[b]);
            }
        } else {
            for (int k = tid; k < cnt; k += kThreads) {
                s_idx[b][0][k] = __ldg(su + k);
                s_idx[b][1][k] = __ldg(si + k);
                s_idx[b][2][k] = __ldg(sj + k);
            }
            __syncthreads();
            if (tid == 0) mbar_arrive(&s_bar[b]);
        }
    };

    for (long long s = 0; s < p.n_steps; ++s) {
        const long long step = p.first_step + s;
        const long long base = p.step_offsets ? __ldg(p.step_offsets + step) : step * p.batch;
        const long long nb = p.step_offsets ? __ldg(p.step_offsets + step + 1) - base : min(p.batch, p.n - base);
        const long long ntiles = (nb + tile - 1) / tile;
        double *acc = hdr->acc[s & 1];
        const bool has_reg = (p.reg1 != 0.f) || (p.reg2 != 0.f);
        if constexpr (XCH::kActive) xch.begin_step(p, s, acc);   // item-side accumulators of this step's parity

        // ------------------------------------------------------------ phase 1
        if (p.phases & 1) {
        if (tid < 8 * (kThreads / 32)) (&s_red[0][0])[tid] = 0.0;   // per-warp fp64 accumulators of this step
        __syncthreads();
        int buf = 0;
        long long t_i = blockIdx.x;
        if (t_i < ntiles) stage(base + t_i * tile, (int)min((long long)tile, nb - t_i * tile), 0);
        for (; t_i < ntiles; t_i += gridDim.x) {
            long long t_n = t_i + gridDim.x;
            if (t_n < ntiles) stage(base + t_n * tile, (int)min((long long)tile, nb - t_n * tile), buf ^ 1);
            if (buf == 0) { mbar_wait(&s_bar[0], par0); par0 ^= 1; } else { mbar_wait(&s_bar[1], par1); par1 ^= 1; }
            const int cnt = (int)min((long long)tile, nb - t_i * tile);
            const int32_t *xu = s_idx[buf][0], *xi = s_idx[buf][1], *xj = s_idx[buf][2];
            float t_loss = 0.f, t_l1u = 0.f, t_l1i = 0.f, t_l1j = 0.f, t_s2u = 0.f, t_s2i = 0.f, t_s2j = 0.f, t_gb0 = 0.f;

            for (int tb = 0; tb < cnt; tb += GROUPS * UNR) {
                Row<VEC, W, NCH> rp[UNR], rqi[UNR], rqj[UNR];
                int iu[UNR], ii[UNR], ij[UNR];
                RowOff ou[UNR], oi[UNR], oj[UNR];   // element offsets of the three rows (tables and accumulators alike)
                float lab[UNR];
                bool ok[UNR];
#pragma unroll
                for (int r = 0; r < UNR; ++r) {
                    int t = tb + r * GROUPS + group;
                    ok[r] = t < cnt;
                    iu[r] = ok[r] ? xu[t] : 0;
                    ii[r] = ok[r] ? xi[t] : 0;
                    ij[r] = ok[r] ? xj[t] : 0;
                    lab[r] = 0.f;
                    if (pw) {                       // label = batch[2].float() (MFRecommender.py:76); the j row stays zero
                        lab[r] = (float)ij[r];
                        ij[r] = 0;
                    }
                    if (!LEAN && p.neg_row_ptr != nullptr && ok[r]) {
                        const long long gt = base + t_i * tile + t;            // position of the triple in the planes
                        ij[r] = draw_negative(p, iu[r], (unsigned long long)gt, (unsigned long long)step);
                        if (p.neg_out != nullptr && gl == 0) p.neg_out[gt] = ij[r];
                    }
                    ou[r] = (RowOff)iu[r] * (RowOff)F;
                    oi[r] = (RowOff)ii[r] * (RowOff)F;
                    oj[r] = (RowOff)ij[r] * (RowOff)F;
                    rp[r] = load_row<VEC, W, NCH>(p.P + ou[r], gl, chunks, ok[r]);
                    rqi[r] = load_row<VEC, W, NCH>(p.Q + oi[r], gl, chunks, ok[r]);
                    rqj[r] = load_row<VEC, W, NCH>(p.Q + oj[r], gl, chunks, ok[r] && !pw);
                }
                // scores of the UNR triples of this group (every lane of the group ends up with the same values)
                float ps[UNR], ns[UNR], cs[UNR], cn[UNR];
#pragma unroll
                for (int r = 0; r < UNR; ++r) {
                    ps[r] = dot_rows<VEC, W, NCH>(rp[r], rqi[r]);
                    ns[r] = dot_rows<VEC, W, NCH>(rp[r], rqj[r]);
                    if (GEN && p.bias != nullptr) {   // FM: pred += (u_bias(user) + i_bias(item)) + bias_  (FMRecommender.py:66-67)
                        const float ub = __ldcg(p.bias + iu[r]), b0 = __ldcg(p.bias + p.U + p.I);
                        ps[r] += (ub + __ldcg(p.bias + p.U + ii[r])) + b0;
                        ns[r] += (ub + __ldcg(p.bias + p.U + ij[r])) + b0;
                    }
                    if (pw) ns[r] = lab[r];         // pair_loss receives the label in place of the negative score
                }
                // The scalar chain (sigmoid -> log -> coefficient, ~40 instructions) would be replayed by all W lanes for
                // each of the UNR triples; instead lane gl evaluates it ONCE, for triple (gl % UNR) of its group, and the
                // coefficients d(loss)/d(pos), d(loss)/d(neg) are handed round with shuffles.
                auto pair_loss = [&](float pos, float neg, float &c_pos, float &c_neg) -> float {
                    if (GEN && p.loss == DRB_LOSS_CL) {     // BCEWithLogitsLoss(sum): (1-y) x - log_sigmoid(x), neg = y
                        const float z = expf(-fabsf(pos));
                        const float logsig = fminf(pos, 0.f) - log1pf(z);
                        const float dls = pos < 0.f ? 1.f - z / (1.f + z) : z / (1.f + z);
                        c_pos = (1.f - neg) - dls;
                        c_neg = 0.f;
                        return (1.f - neg) * pos - logsig;
                    }
                    if (GEN && p.loss == DRB_LOSS_SL) {     // MSELoss(sum): (x - y)^2, neg = y
                        const float d = pos - neg;
                        c_pos = 2.f * d;
                        c_neg = 0.f;
                        return d * d;
                    }
                    if (GEN && p.loss == DRB_LOSS_HL) {     // clamp(1 - (pos - neg), min=0); clamp's backward passes at equality
                        const float m = 1.f - (pos - neg);
                        c_pos = (m >= 0.f) ? -1.f : 0.f;
                        c_neg = -c_pos;
                        return m > 0.f ? m : 0.f;
                    }
                    if (GEN && p.loss == DRB_LOSS_TL) {     // sigmoid(neg - pos) + sigmoid(neg^2)
                        const float s1 = 1.f / (1.f + expf(-(neg - pos))), s2 = 1.f / (1.f + expf(-(neg * neg)));
                        c_pos = -(s1 * (1.f - s1));
                        c_neg = s1 * (1.f - s1) + s2 * (1.f - s2) * 2.f * neg;
                        return s1 + s2;
                    }
                    const float x = pos - neg;
                    const float sg = 1.f / (1.f + expf(-x));
                    c_pos = -(sg * (1.f - sg)) / (1e-10f + sg);
                    c_neg = -c_pos;
                    return -logf(1e-10f + sg);
                };
                if constexpr (W >= UNR) {
                    float p_own = ps[0], n_own = ns[0];
                    bool ok_own = ok[0];
#pragma unroll
                    for (int r = 1; r < UNR; ++r)
                        if ((gl % UNR) == r) { p_own = ps[r]; n_own = ns[r]; ok_own = ok[r]; }
                    float cp_own, cn_own;
                    const float l_own = pair_loss(p_own, n_own, cp_own, cn_own);
                    if (gl < UNR && ok_own) t_loss += l_own;
#pragma unroll
                    for (int r = 0; r < UNR; ++r) {
                        cs[r] = __shfl_sync(0xffffffffu, cp_own, (lane - gl) + r);
                        cn[r] = GEN ? __shfl_sync(0xffffffffu, cn_own, (lane - gl) + r) : -cs[r];
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < UNR; ++r) {
                        const float l = pair_loss(ps[r], ns[r], cs[r], cn[r]);
                        if (gl == 0 && ok[r]) t_loss += l;
                    }
                }
#pragma unroll
                for (int r = 0; r < UNR; ++r) {
                    if (!ok[r]) continue;
                    const float c = cs[r];
                    if (has_reg) {
                        float l1u = 0, l1i = 0, l1j = 0, s2u = 0, s2i = 0, s2j = 0;
                        Row<VEC, W, NCH> nu_ = rp[r], ni_ = rqi[r], nj_ = rqj[r];
                        if (!LEAN && p.Pn != nullptr) {   // regulariser on the ego rows (LightGCNRecommender.py:145-146,159)
                            nu_ = load_row<VEC, W, NCH>(p.Pn + ou[r], gl, chunks, true);
                            ni_ = load_row<VEC, W, NCH>(p.Qn + oi[r], gl, chunks, true);
                            nj_ = load_row<VEC, W, NCH>(p.Qn + oj[r], gl, chunks, true);
                        }
#pragma unroll
                        for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
                            for (int e = 0; e < VEC; ++e) {
                                float a = nu_.c[ch].v[e], b = ni_.c[ch].v[e], d = nj_.c[ch].v[e];
                                l1u += fabsf(a); s2u = fmaf(a, a, s2u);
                                l1i += fabsf(b); s2i = fmaf(b, b, s2i);
                                l1j += fabsf(d); s2j = fmaf(d, d, s2j);
                            }
                        t_l1u += l1u; t_l1i += l1i; t_l1j += l1j;
                        t_s2u += s2u; t_s2i += s2i; t_s2j += s2j;
                    }
                    if (p.apply) {
#pragma unroll
                        for (int ch = 0; ch < NCH; ++ch) {
                            int cc = gl + ch * W;
                            if (cc >= chunks) continue;
                            Vec<VEC> gu, gi, gj;
#pragma unroll
                            for (int e = 0; e < VEC; ++e) {
                                if (!GEN || p.loss == DRB_LOSS_BPR) {   // c_neg == -c_pos: the reference's BPR arithmetic
                                    gu.v[e] = c * (rqi[r].c[ch].v[e] - rqj[r].c[ch].v[e]);
                                    gi.v[e] = c * rp[r].c[ch].v[e];
                                    gj.v[e] = -gi.v[e];
                                } else {
                                    gu.v[e] = c * rqi[r].c[ch].v[e] + cn[r] * rqj[r].c[ch].v[e];
                                    gi.v[e] = c * rp[r].c[ch].v[e];
                                    gj.v[e] = cn[r] * rp[r].c[ch].v[e];
                                }
                            }
                            if (GEN && p.det) {
#pragma unroll
                                for (int e = 0; e < VEC; ++e) {
                                    det_red(p.ws.gP64 + ou[r] + cc * VEC + e, gu.v[e]);
                                    det_red(p.ws.gQ64 + oi[r] + cc * VEC + e, gi.v[e]);
                                    if (!pw) det_red(p.ws.gQ64 + oj[r] + cc * VEC + e, gj.v[e]);
                                }
                            } else {
                                red_row<VEC>(p.ws.gP + ou[r] + cc * VEC, gu);
                                red_row<VEC>(p.ws.gQ + oi[r] + cc * VEC, gi);
                                if (!pw) red_row<VEC>(p.ws.gQ + oj[r] + cc * VEC, gj);
                            }
                        }
                        if (gl == 0) {
                            if (GEN && p.shared) red_add_u64(p.ws.cntI + iu[r], 1ull);   // the target is an item row too
                            else red_add_u32(p.ws.cntU + iu[r], 1u);
                            red_add_u64(p.ws.cntI + ii[r], 1ull);
                            if (!pw) red_add_u64(p.ws.cntI + ij[r], 1ull << 32);
                            if (GEN && p.bias != nullptr) {   // d loss / d (u_bias, i_bias, bias_): no regulariser (:76-95)
                                const float cboth = pw ? c : c + cn[r];
                                asm volatile("red.relaxed.gpu.global.add.f32 [%0], %1;" ::"l"(p.ws.gB + iu[r]), "f"(cboth) : "memory");
                                asm volatile("red.relaxed.gpu.global.add.f32 [%0], %1;" ::"l"(p.ws.gB + p.U + ii[r]), "f"(c) : "memory");
                                if (!pw)
                                    asm volatile("red.relaxed.gpu.global.add.f32 [%0], %1;" ::"l"(p.ws.gB + p.U + ij[r]), "f"(cn[r]) : "memory");
                                t_gb0 += cboth;
                            }
                        }
                    }
                }
            }
            // per-thread fp32 partials cover <= tile/GROUPS triples: warp-reduce, widen to fp64 in smem
            {
                float tv[8] = {t_loss, t_l1u, t_l1i, t_l1j, t_s2u, t_s2i, t_s2j, t_gb0};
                const int nv = has_reg ? 7 : 1;
                for (int k = 0; k < 8; ++k) {
                    if (k >= nv && !(GEN && k == 7 && p.bias != nullptr)) continue;
                    float v = tv[k];
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                    if (lane == 0) s_red[k][warp] += (double)v;
                }
            }
            __syncthreads();  // tile buffer free for re-staging
            buf ^= 1;
        }
        // CTA reduction of the 7 partial sums -> one fp64 atomic each
        __syncthreads();
        if (tid < (has_reg ? 7 : 1) || (GEN && tid == 7 && p.bias != nullptr)) {
            double v = 0;
            for (int w = 0; w < kThreads / 32; ++w) v += s_red[tid][w];
            if (GEN && p.det) {
                if (v != 0.0) red_add_u64(reinterpret_cast<unsigned long long *>(p.ws.accfx + tid),
                                          (unsigned long long)__double2ll_rn(v * kDetAccScale));
            } else if (v != 0.0) {
                atomicAdd(&acc[tid], v);
            }
        }
        }  // phase 1
        if (p.phases == 3) grid_barrier(&hdr->barrier, epoch);
        if (!(p.phases & 2)) break;   // split mode: the host reduces gQ / counters / acc across ranks now
        if (GEN && p.det) {
            // fixed-point sums -> the fp32 accumulators phase 2 reads (one rounding per element, whatever order the atomics took)
            const long long gsz = (long long)gridDim.x * kThreads, gt = (long long)blockIdx.x * kThreads + tid;
            const long long nP = (long long)p.U * F, nQ = (long long)p.I * F;
            for (long long k = gt; k < nP + nQ; k += gsz) {
                long long *src = k < nP ? p.ws.gP64 + k : p.ws.gQ64 + (k - nP);
                const long long v = __ldcg(src);
                if (v != 0) {
                    __stcg((k < nP ? p.ws.gP + k : p.ws.gQ + (k - nP)), (float)((double)v / kDetScale));
                    __stcg(src, 0ll);
                }
            }
            if (gt < 8) {
                acc[gt] = (double)__ldcg(p.ws.accfx + gt) / kDetAccScale;
                __stcg(p.ws.accfx + gt, 0ll);
            }
            grid_barrier(&hdr->barrier, epoch);
        }
        if constexpr (XCH::kActive) {
            // rendezvous with the other ranks; acc[0..7] become the GLOBAL sums (identical on every rank)
            if (!xch.after_phase1(p, s, acc, epoch)) break;
        }

        // ------------------------------------------------------------ phase 2
        double bpr, l1u, l1i, l1j, s2u, s2i, s2j;
        {
            const volatile double *va = acc;
            bpr = va[0]; l1u = va[1]; l1i = va[2]; l1j = va[3]; s2u = va[4]; s2i = va[5]; s2j = va[6];
        }
        double nu = sqrt(s2u), ni = sqrt(s2i), nj = sqrt(s2j);
        // fp32 assembly of the scalar loss, in the reference's order (MFRecommender.py:88-95)
        float loss = (float)bpr;
        loss += p.reg1 * ((float)l1i + (float)l1j);
        loss += p.reg2 * ((float)ni + (float)nj);
        loss += p.reg1 * (float)l1u;
        loss += p.reg2 * (float)nu;
        if (blockIdx.x == 0 && tid == 0) p.step_loss[s] = (double)loss;
        if constexpr (!XCH::kActive)
            if (blockIdx.x == 0 && tid < 8) hdr->acc[(s + 1) & 1][tid] = 0.0;  // recycle the other accumulator
        if (isnan(loss)) {
            if (blockIdx.x == 0 && tid == 0) {
                hdr->status = DRB_ERR_NAN_LOSS;
                hdr->nan_step = step;
            }
            break;  // uniform across the grid: every CTA computed the same loss
        }
        if (p.apply) {
            Norms nm;
            nm.inv_u = nu > 0 ? (float)(1.0 / nu) : 0.f;
            nm.inv_i = ni > 0 ? (float)(1.0 / ni) : 0.f;
            nm.inv_j = nj > 0 ? (float)(1.0 / nj) : 0.f;
            AdamCoef ac;
            ac.step_size = 0.f;
            ac.bc2_sqrt = 1.f;
            if (p.opt == DRB_OPT_ADAM) {
                double t = (double)(p.adam_step0 + s + 1);
                ac.step_size = (float)((double)p.lr / (1.0 - pow((double)p.beta1, t)));
                ac.bc2_sqrt = (float)sqrt(1.0 - pow((double)p.beta2, t));
            }
            const bool dense = p.dense_hint >= 0 ? (p.dense_hint != 0)
                                                 : ((p.opt != DRB_OPT_SGD) || (3 * nb >= ((long long)p.U + p.I) / 4));
            if constexpr (XCH::kActive) {
                // this rank's item slice: reduce the ranks' accumulators, update, broadcast the new rows; then the local user
                // rows are swept below with the item half switched off (p.I = 0 inside the policy's copy of the parameters)
                xch.template item_slice<VEC, W, NCH>(p, s, nm, ac, gl, group, GROUPS, chunks, epoch);
            }
            if (dense || p.opt != DRB_OPT_SGD) {   // stateful optimisers always sweep (claim mode is SGD only)
                if (p.opt == DRB_OPT_SGD)
                    dense_sweep<VEC, W, NCH, DRB_OPT_SGD, XCH::kActive>(p, nm, ac, gl, group, GROUPS, chunks);
                else if (p.opt == DRB_OPT_ADAM)
                    dense_sweep<VEC, W, NCH, DRB_OPT_ADAM, XCH::kActive>(p, nm, ac, gl, group, GROUPS, chunks);
                else if constexpr (GEN) {          // launch_steps routes these two to the GEN instantiation
                    if (p.opt == DRB_OPT_ADAGRAD)
                        dense_sweep<VEC, W, NCH, DRB_OPT_ADAGRAD>(p, nm, ac, gl, group, GROUPS, chunks);
                    else
                        dense_sweep<VEC, W, NCH, DRB_OPT_RMSPROP>(p, nm, ac, gl, group, GROUPS, chunks);
                }
            } else {
                // claim mode (SGD only): the first group to swap a row's counter to zero applies it
                for (long long t0 = (long long)blockIdx.x * tile; t0 < nb; t0 += (long long)gridDim.x * tile) {
                    const int cnt = (int)min((long long)tile, nb - t0);
                    for (int tb = 0; tb < cnt; tb += GROUPS) {
                        int t = tb + group;
                        bool ok = t < cnt;
                        int u = 0, i = 0, j = 0;
                        if (ok) {
                            u = __ldg(p.bu + base + t0 + t);
                            i = __ldg(p.bi + base + t0 + t);
                            j = pw ? i : __ldg(p.bj + base + t0 + t);   // point-wise: that plane holds labels
                            if (GEN && p.shared) j = u;                  // shared table: the target is claimed as an item row
                        }
                        unsigned cu = 0;
                        unsigned long long ci = 0, cj = 0;
                        if (ok && gl == 0) {
                            if (!(GEN && p.shared)) cu = atomicExch(p.ws.cntU + u, 0u);
                            ci = atomicExch(p.ws.cntI + i, 0ull);
                            cj = atomicExch(p.ws.cntI + j, 0ull);
                        }
                        cu = __shfl_sync(0xffffffffu, cu, gw * W);
                        ci = __shfl_sync(0xffffffffu, ci, gw * W);
                        cj = __shfl_sync(0xffffffffu, cj, gw * W);
                        if (cu != 0) {
                            size_t o = (size_t)u * F;
                            apply_row<VEC, W, NCH, DRB_OPT_SGD>(p.P + o, p.ws.gP + o, nullptr, nullptr, gl, chunks, (float)cu,
                                                                nm.inv_u, 0.f, 0.f, p, ac, true);
                        }
                        if (ci != 0) {
                            size_t o = (size_t)i * F;
                            apply_row<VEC, W, NCH, DRB_OPT_SGD>(p.Q + o, p.ws.gQ + o, nullptr, nullptr, gl, chunks,
                                                                (float)(unsigned)(ci & 0xffffffffull), nm.inv_i,
                                                                (float)(unsigned)(ci >> 32), nm.inv_j, p, ac, true);
                        }
                        if (cj != 0) {
                            size_t o = (size_t)j * F;
                            apply_row<VEC, W, NCH, DRB_OPT_SGD>(p.Q + o, p.ws.gQ + o, nullptr, nullptr, gl, chunks,
                                                                (float)(unsigned)(cj & 0xffffffffull), nm.inv_i,
                                                                (float)(unsigned)(cj >> 32), nm.inv_j, p, ac, true);
                        }
                    }
                }
            }
        }
        if (GEN && p.apply && p.bias != nullptr) {
            // FM's U + I + 1 first-order scalars: the same optimiser switch, no regulariser; the accumulator is cleared
            const double gb0 = ((const volatile double *)acc)[7];
            float step_size = 0.f, bc2_sqrt = 1.f;
            if (p.opt == DRB_OPT_ADAM) {
                double t = (double)(p.adam_step0 + s + 1);
                step_size = (float)((double)p.lr / (1.0 - pow((double)p.beta1, t)));
                bc2_sqrt = (float)sqrt(1.0 - pow((double)p.beta2, t));
            }
            const long long nbias = (long long)p.U + p.I + 1;
            for (long long k = (long long)blockIdx.x * kThreads + tid; k < nbias; k += (long long)gridDim.x * kThreads) {
                const float g = (k == nbias - 1) ? (float)gb0 : __ldcg(p.ws.gB + k);
                float th = __ldcg(p.bias + k);
                if (p.opt == DRB_OPT_SGD) {
                    th = th - p.lr * g;
                } else if (p.opt == DRB_OPT_ADAGRAD) {
                    const float ss = __ldcg(p.ws.mB + k) + g * g;
                    th = th - p.lr * (g / (sqrtf(ss) + 1e-10f));
                    __stcg(p.ws.mB + k, ss);
                } else if (p.opt == DRB_OPT_RMSPROP) {
                    const float sq = __ldcg(p.ws.mB + k) * 0.99f + (1.f - 0.99f) * g * g;
                    th = th - p.lr * (g / (sqrtf(sq) + 1e-8f));
                    __stcg(p.ws.mB + k, sq);
                } else {
                    float mm = __ldcg(p.ws.mB + k), vv = __ldcg(p.ws.vB + k);
                    mm = mm + (g - mm) * (1.f - p.beta1);
                    vv = vv * p.beta2 + (1.f - p.beta2) * g * g;
                    th = th - step_size * (mm / (sqrtf(vv) / bc2_sqrt + p.eps));
                    __stcg(p.ws.mB + k, mm);
                    __stcg(p.ws.vB + k, vv);
                }
                __stcg(p.bias + k, th);
                if (k != nbias - 1 && g != 0.f) __stcg(p.ws.gB + k, 0.f);
            }
        }
        if constexpr (XCH::kActive) {
            if (!xch.end_step(p, s, epoch)) break;   // every rank's item slice has landed in this rank's replica
        } else {
            if (s + 1 < p.n_steps) grid_barrier(&hdr->barrier, epoch);
        }
    }
}

template <int VEC, int W, int NCH, bool GEN>
__global__ void __launch_bounds__(kThreads, DRB_MINB) mf_bpr_steps_kernel(StepParams p)
{
    NoExchange x;
    bpr_steps_body<VEC, W, NCH, GEN, NoExchange>(p, x);
}

template <int VEC, int W, int NCH>
__global__ void __launch_bounds__(kThreads, DRB_MINB) mf_bpr_steps_lean_kernel(StepParams p)
{
    NoExchange x;
    bpr_steps_body<VEC, W, NCH, false, NoExchange, true>(p, x);
}

// the conditions under which the lean body computes what the general one does
inline bool step_params_lean(const StepParams &p)
{
    return p.loss == DRB_LOSS_BPR && p.opt <= DRB_OPT_ADAM && p.bias == nullptr && p.det == 0 && p.Pn == nullptr &&
           p.Qn == nullptr && p.neg_row_ptr == nullptr && (unsigned long long)p.U * (unsigned)p.F < (1ull << 32) &&
           (unsigned long long)p.I * (unsigned)p.F < (1ull << 32);
}


}  // namespace drb
