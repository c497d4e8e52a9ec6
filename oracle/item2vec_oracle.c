/* item2vec_oracle.c -- plain-C restatement of Item2Vec for the tests (TEST INFRASTRUCTURE ONLY, like bpr_oracle.c).
 *
 *   orc_sgns_sample      SkipGramNegativeSampler.sampling() (daisy/utils/sampler.py:130-155): sequential, on numpy's legacy
 *                        MT19937 state, one np.random.choice(cands, size=c) per target position
 *   orc_item2vec_step    one step of Item2Vec.calc_loss + backward + optimizer.step (Item2VecRecommender.py:62-69,
 *                        AbstractRecommender.py:48-67,112-128): BCEWithLogitsLoss(sum) on <Q[t], Q[c]>, fp64 scores and
 *                        gradients, the fp32 torch optimiser updates on every row of the dense table
 *   orc_item2vec_user_embed  user_embedding[u] = sum of Q over the user's sorted train row (:56-60), fp32 in row order
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* numpy legacy MT19937: state = 624 key words + position */
static uint32_t mt_next(uint32_t *st)
{
    uint32_t *mt = st;
    if (st[624] >= 624) {
        const uint32_t UP = 0x80000000u, LO = 0x7fffffffu, MAG = 0x9908b0dfu;
        for (int k = 0; k < 624; ++k) {
            uint32_t y = (mt[k] & UP) | (mt[(k + 1) % 624] & LO);
            mt[k] = mt[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? MAG : 0u);
        }
        st[624] = 0;
    }
    uint32_t y = mt[st[624]++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

/* RandomState.randint(0, n) as np.random.choice(a, size) draws it: masked rejection, n == 1 consumes no word */
static uint32_t mt_bounded(uint32_t *st, uint32_t n)
{
    uint32_t mx = n - 1u, mask = mx, v;
    if (mx == 0u) return 0u;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    while ((v = mt_next(st) & mask) > mx) {}
    return v;
}

/* the k-th smallest item of [0, I) missing from the sorted row col[b, e) */
static int32_t kth_missing(const int32_t *col, int64_t b, int64_t e, int32_t k)
{
    int32_t item = k;
    for (int64_t s = b; s < e && col[s] <= item; ++s) ++item;
    return item;
}

/* users / items [n]: the df rows.  rows_out [cap, 3] int64.  Returns the row count T, -1 when cap is too small, -2 when a
 * position with context has an empty complement (numpy's ValueError; the state is left where numpy leaves it). */
int64_t orc_sgns_sample(uint32_t *st, const int32_t *users, const int32_t *items, int64_t n, const int64_t *row_ptr,
                        const int32_t *col, int32_t I, int32_t w, int64_t *rows_out, int64_t cap)
{
    int64_t *order = (int64_t *)malloc(sizeof(int64_t) * (size_t)(n > 0 ? n : 1));
    int32_t umax = -1;
    for (int64_t p = 0; p < n; ++p) if (users[p] > umax) umax = users[p];
    int64_t *start = (int64_t *)calloc((size_t)umax + 2, sizeof(int64_t));
    for (int64_t p = 0; p < n; ++p) start[users[p] + 1]++;
    for (int32_t u = 0; u <= umax; ++u) start[u + 1] += start[u];
    int64_t *fill = (int64_t *)malloc(sizeof(int64_t) * ((size_t)umax + 1));
    for (int32_t u = 0; u <= umax; ++u) fill[u] = start[u];
    for (int64_t p = 0; p < n; ++p) order[fill[users[p]]++] = p;       /* stable: df order inside a user */
    int64_t T = 0;
    for (int32_t u = 0; u <= umax && T >= 0; ++u) {
        const int64_t s = start[u], L = start[u + 1] - s;
        const int64_t deg = row_ptr[u + 1] - row_ptr[u];
        for (int64_t i = 0; i < L && T >= 0; ++i) {
            const int64_t t = items[order[s + i]];
            int64_t c = 0;
            for (int64_t j = i - w; j <= i + w && j < L; ++j) {
                if (j < 0 || j == i) continue;
                if (T >= cap) { T = -1; break; }
                rows_out[3 * T] = t; rows_out[3 * T + 1] = items[order[s + j]]; rows_out[3 * T + 2] = 1;
                ++T; ++c;
            }
            if (T < 0) break;
            if (c > 0 && (int64_t)I - deg <= 0) { T = -2; break; }
            for (int64_t k = 0; k < c; ++k) {
                if (T >= cap) { T = -1; break; }
                const int32_t r = (int32_t)mt_bounded(st, (uint32_t)((int64_t)I - deg));
                rows_out[3 * T] = t; rows_out[3 * T + 1] = kth_missing(col, row_ptr[u], row_ptr[u + 1], r);
                rows_out[3 * T + 2] = 0;
                ++T;
            }
        }
    }
    free(order); free(start); free(fill);
    return T;
}

/* opt: 0 SGD, 1 Adam, 2 Adagrad, 3 RMSprop (torch defaults).  m / v: optimiser state [I*F] (Adagrad / RMSprop: m only).
 * step_count: the optimiser step this is (1-based, Adam bias correction).  apply = 0: loss only.  Returns the fp64 sum. */
double orc_item2vec_step(float *Q, int32_t I, int32_t F, const int32_t *bt, const int32_t *bc, const int32_t *bl, int64_t B,
                         int32_t opt, float lr, float beta1, float beta2, float eps, float *m, float *v, int64_t step_count,
                         int32_t apply)
{
    double *g = (double *)calloc((size_t)I * F, sizeof(double));
    double loss = 0.0;
    for (int64_t b = 0; b < B; ++b) {
        const float *qt = Q + (size_t)bt[b] * F, *qc = Q + (size_t)bc[b] * F;
        double x = 0.0;
        for (int f = 0; f < F; ++f) x += (double)qt[f] * qc[f];
        const double y = (double)bl[b];
        loss += (x > 0 ? x : 0) - x * y + log1p(exp(-fabs(x)));
        const double d = 1.0 / (1.0 + exp(-x)) - y;              /* d loss / d x */
        for (int f = 0; f < F; ++f) {
            g[(size_t)bt[b] * F + f] += d * qc[f];
            g[(size_t)bc[b] * F + f] += d * qt[f];
        }
    }
    if (apply) {
        const double bc1 = 1.0 - pow((double)beta1, (double)step_count);
        const double bc2 = 1.0 - pow((double)beta2, (double)step_count);
        const float step_size = (float)(lr / bc1), bc2_sqrt = (float)sqrt(bc2);
        for (size_t e = 0; e < (size_t)I * F; ++e) {
            const float gg = (float)g[e];
            if (opt == 0) {
                Q[e] = Q[e] - lr * gg;
            } else if (opt == 1) {
                m[e] = m[e] + (gg - m[e]) * (1.f - beta1);
                v[e] = v[e] * beta2 + (1.f - beta2) * gg * gg;
                Q[e] = Q[e] - step_size * (m[e] / (sqrtf(v[e]) / bc2_sqrt + eps));
            } else if (opt == 2) {
                m[e] = m[e] + gg * gg;
                Q[e] = Q[e] - lr * (gg / (sqrtf(m[e]) + 1e-10f));
            } else {
                m[e] = m[e] * 0.99f + (1.f - 0.99f) * gg * gg;
                Q[e] = Q[e] - lr * (gg / (sqrtf(m[e]) + 1e-8f));
            }
        }
    }
    free(g);
    return loss;
}

void orc_item2vec_user_embed(const int64_t *row_ptr, const int32_t *col, const float *Q, int32_t U, int32_t F, float *P)
{
    for (int32_t u = 0; u < U; ++u) {
        if (row_ptr[u + 1] == row_ptr[u]) continue;
        for (int f = 0; f < F; ++f) {
            float acc = 0.f;
            for (int64_t s = row_ptr[u]; s < row_ptr[u + 1]; ++s) acc += Q[(size_t)col[s] * F + f];
            P[(size_t)u * F + f] = acc;
        }
    }
}
