// sampler.cu -- pair-wise negative sampler of daisyRec on the device.
//
// Stands behind BasicNegtiveSampler.sampling(), uniform + BPR branch
// (daisy/utils/sampler.py:55-103).  The reference, per user, materialises
// setdiff1d(arange(item_num), past_inter) (O(item_num) each, O(U*I) total) and indexes it with
// num_ng bounded draws of numpy's legacy MT19937.  Here:
//   * the draws  k = randint(0, item_num - deg(u))  are the only sequential part (the number of
//     32-bit words a draw consumes depends on rejections) -> host, O(U*G) words
//     (drb_sampler_draw_mt19937), or counter-based Philox on the device in throughput mode;
//   * the k-th element of the sorted complement is found WITHOUT building the complement:
//     item = k + #{s : col[s] - s <= k} over the user's sorted CSR row (col[s]-s is
//     non-decreasing, so one binary search) -> device, one thread per (u, g);
//   * the explode to int32 [nnz*G, 3] rows (sampler.py:91,99-101) -> device, one thread per row.
#include "common.cuh"

namespace drb {

// ---------------------------------------------------------------- numpy legacy MT19937 (host)
struct Mt {
    uint32_t *key;  // 624 words
    uint32_t *pos;
    void regen()
    {
        const uint32_t UP = 0x80000000u, LO = 0x7fffffffu, MAG = 0x9908b0dfu;
        uint32_t *mt = key;
        int k = 0;
        for (; k < 624 - 397; ++k) {
            uint32_t y = (mt[k] & UP) | (mt[k + 1] & LO);
            mt[k] = mt[k + 397] ^ (y >> 1) ^ (-(int32_t)(y & 1u) & MAG);
        }
        for (; k < 623; ++k) {
            uint32_t y = (mt[k] & UP) | (mt[k + 1] & LO);
            mt[k] = mt[k - 227] ^ (y >> 1) ^ (-(int32_t)(y & 1u) & MAG);
        }
        uint32_t y = (mt[623] & UP) | (mt[0] & LO);
        mt[623] = mt[396] ^ (y >> 1) ^ (-(int32_t)(y & 1u) & MAG);
        *pos = 0;
    }
    uint32_t next()
    {
        if (*pos >= 624) regen();
        uint32_t y = key[(*pos)++];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= y >> 18;
        return y;
    }
    // RandomState.random_sample(): 53-bit double from two words (legacy mt19937_next_double)
    double uniform01()
    {
        uint32_t a = next() >> 5, b = next() >> 6;
        return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
    }
    // RandomState.randint(0, n): masked rejection on 32-bit words; n == 1 consumes nothing
    uint32_t bounded(uint32_t n)
    {
        uint32_t mx = n - 1u;
        if (mx == 0u) return 0u;
        uint32_t mask = mx;
        mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
        uint32_t v;
        while ((v = next() & mask) > mx) {}
        return v;
    }
};

__global__ void draw_philox_kernel(uint64_t seed, uint64_t offset, const int64_t *__restrict__ row_ptr, int U, int I, int G,
                                   int32_t *__restrict__ draws, int32_t *__restrict__ bad_user)
{
    long long total = (long long)U * G;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        int u = (int)(idx / G);
        long long deg = row_ptr[u + 1] - row_ptr[u];
        long long n = (long long)I - deg;
        if (n <= 0) {
            atomicMin(bad_user, u);
            draws[idx] = 0;
            continue;
        }
        uint32_t mx = (uint32_t)(n - 1), mask = mx;
        mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
        uint32_t v = 0;
        bool done = (mx == 0);
        for (uint32_t attempt = 0; !done; ++attempt) {  // masked rejection: exact uniform, <2 words expected
            uint32_t c[4] = {(uint32_t)idx, (uint32_t)((uint64_t)idx >> 32), (uint32_t)offset + attempt,
                             (uint32_t)(offset >> 32)};
            philox4x32(c, (uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
            for (int w = 0; w < 4 && !done; ++w) {
                v = c[w] & mask;
                done = v <= mx;
            }
        }
        draws[idx] = (int32_t)v;
    }
}

// the k-th smallest item missing from the sorted row col[b, e): k + #{s : col[s] - s <= k} (col[s] - s is non-decreasing,
// so one binary search)
__device__ __forceinline__ int kth_complement(const int32_t *__restrict__ col, long long b, long long e, int k)
{
    long long lo = 0, hi = e - b;  // first s with col[s]-s > k
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if ((long long)__ldg(col + b + mid) - mid <= (long long)k) lo = mid + 1; else hi = mid;
    }
    return k + (int)lo;
}

// js[u,g] = k-th smallest item not in the user's sorted row (k = draws[u,g])
__global__ void kth_complement_kernel(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ col,
                                      const int32_t *__restrict__ draws, int U, int G, int32_t *__restrict__ js)
{
    long long total = (long long)U * G;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        int u = (int)(idx / G);
        js[idx] = kth_complement(col, row_ptr[u], row_ptr[u + 1], draws[idx]);
    }
}

// variable number of draws per row: row m owns draws[offsets[m] .. offsets[m+1])
__global__ void kth_complement_var_kernel(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ col,
                                          const int64_t *__restrict__ offsets, const int32_t *__restrict__ draws,
                                          long long rows, int32_t *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long m = warp; m < rows; m += nwarps) {          // one warp per row
        long long b = row_ptr[m], e = row_ptr[m + 1];
        for (long long d = offsets[m] + lane; d < offsets[m + 1]; d += 32) out[d] = kth_complement(col, b, e, draws[d]);
    }
}

__global__ void explode_kernel(const int32_t *__restrict__ coo_u, const int32_t *__restrict__ coo_i, long long nnz,
                               const int32_t *__restrict__ js, int G, int32_t *__restrict__ triples)
{
    long long total = nnz * G;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        long long r = idx / G;
        int g = (int)(idx - r * G);
        int u = __ldg(coo_u + r);
        int32_t *t = triples + 3 * idx;
        t[0] = u;
        t[1] = __ldg(coo_i + r);
        t[2] = __ldg(js + (long long)u * G + g);
    }
}

// popularity-mixed table (sampler.py:64-81): columns [0, un) = k-th complement of a uniform rank, columns
// [un, un+on) = searchsorted(cdf, x, side='right') of a uniform double (RandomState.choice(p=...))
__global__ void assemble_mixed_kernel(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ col,
                                      const int32_t *__restrict__ draws, const double *__restrict__ cdf,
                                      const double *__restrict__ u01, int U, int I, int un, int on,
                                      int32_t *__restrict__ js)
{
    const int G = un + on;
    long long total = (long long)U * G;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        int u = (int)(idx / G), g = (int)(idx - (long long)u * G);
        if (g < un) {
            js[idx] = kth_complement(col, row_ptr[u], row_ptr[u + 1], draws[(long long)u * un + g]);
        } else {
            double x = u01[(long long)u * on + (g - un)];
            int lo = 0, hi = I;  // first index with cdf[index] > x
            while (lo < hi) {
                int mid = (lo + hi) >> 1;
                if (__ldg(cdf + mid) <= x) lo = mid + 1; else hi = mid;
            }
            js[idx] = lo;
        }
    }
}

// point-wise explode (sampler.py:93-98): nnz positive rows (u, i, label) then nnz*G negative rows (u, js[u,g], 0)
__global__ void explode_pointwise_kernel(const int32_t *__restrict__ coo_u, const int32_t *__restrict__ coo_i,
                                         const int32_t *__restrict__ label, long long nnz,
                                         const int32_t *__restrict__ js, int G, int32_t *__restrict__ rows)
{
    long long total = nnz * (1 + G);
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        int32_t *t = rows + 3 * idx;
        if (idx < nnz) {
            t[0] = __ldg(coo_u + idx);
            t[1] = __ldg(coo_i + idx);
            t[2] = __ldg(label + idx);
        } else {
            long long n = idx - nnz, r = n / G;
            int g = (int)(n - r * G);
            int u = __ldg(coo_u + r);
            t[0] = u;
            t[1] = __ldg(js + (long long)u * G + g);
            t[2] = 0;
        }
    }
}

// ---------------------------------------------------------------- skip-gram negative sampling (sampler.py:105-160)
// Positions are the df rows grouped stably by user (users ascending, df order inside a user): su / si [n].  Position p sits
// at index i of its user's sequence [s, e); its context window is j in [max(i-w, 0), min(i+w, L-1)] without i.
__device__ __forceinline__ void sgns_segment(const int32_t *__restrict__ su, long long n, long long p, long long &s,
                                             long long &e)
{
    const int u = __ldg(su + p);
    long long lo = 0, hi = p;           // first position of user u
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if (__ldg(su + mid) < u) lo = mid + 1; else hi = mid;
    }
    s = lo;
    lo = p + 1; hi = n;                 // one past its last position
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if (__ldg(su + mid) <= u) lo = mid + 1; else hi = mid;
    }
    e = lo;
}

// count[p] = number of context items of position p (= its number of negatives); bound[p] = I - deg(user), the size of the
// complement its negatives are drawn from
__global__ void sgns_positions_kernel(const int32_t *__restrict__ su, long long n, const int64_t *__restrict__ row_ptr, int I,
                                      int w, int64_t *__restrict__ count, int64_t *__restrict__ bound)
{
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        long long s, e;
        sgns_segment(su, n, p, s, e);
        const long long i = p - s, L = e - s;
        const long long lo = i - w > 0 ? i - w : 0, hi = i + w < L - 1 ? i + w : L - 1;
        count[p] = hi - lo;             // hi - lo + 1 window slots minus the target itself
        const int u = __ldg(su + p);
        bound[p] = (int64_t)I - (row_ptr[u + 1] - row_ptr[u]);
    }
}

// rows[2*off[p] ..] of position p: its c positives [t, seq[j], 1] in ascending j, then its c negatives [t, neg, 0] with
// neg = the draws[off[p] + k]-th item missing from the user's sorted train row
__global__ void sgns_explode_kernel(const int32_t *__restrict__ su, const int32_t *__restrict__ si, long long n, int w,
                                    const int64_t *__restrict__ off, const int64_t *__restrict__ row_ptr,
                                    const int32_t *__restrict__ col, const int32_t *__restrict__ draws,
                                    int32_t *__restrict__ rows)
{
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        long long s, e;
        sgns_segment(su, n, p, s, e);
        const long long i = p - s, L = e - s;
        const long long lo = i - w > 0 ? i - w : 0, hi = i + w < L - 1 ? i + w : L - 1;
        const long long d0 = off[p], c = off[p + 1] - d0;
        const int t = __ldg(si + p), u = __ldg(su + p);
        int32_t *r = rows + 6 * d0;
        for (long long j = lo; j <= hi; ++j) {
            if (j == i) continue;
            r[0] = t; r[1] = __ldg(si + s + j); r[2] = 1;
            r += 3;
        }
        const long long rb = row_ptr[u], re = row_ptr[u + 1];
        for (long long k = 0; k < c; ++k) {
            r[0] = t; r[1] = kth_complement(col, rb, re, __ldg(draws + d0 + k)); r[2] = 0;
            r += 3;
        }
    }
}

}  // namespace drb

using namespace drb;

extern "C" int drb_sgns_positions(const int32_t *d_su, int64_t n, const int64_t *d_row_ptr, int32_t item_num,
                                  int32_t window, int64_t *d_count, int64_t *d_bound, void *stream)
{
    DRB_REQUIRE(d_su && d_row_ptr && d_count && d_bound && n >= 0 && item_num > 0 && window >= 0,
                "sgns_positions: bad arguments");
    if (n == 0) return DRB_OK;
    sgns_positions_kernel<<<grid_size(n, 256), 256, 0, (cudaStream_t)stream>>>(d_su, n, d_row_ptr, item_num, window, d_count,
                                                                               d_bound);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_sgns_explode(const int32_t *d_su, const int32_t *d_si, int64_t n, int32_t window, const int64_t *d_offsets,
                                const int64_t *d_row_ptr, const int32_t *d_col, const int32_t *d_draws, int32_t *d_rows,
                                void *stream)
{
    DRB_REQUIRE(d_su && d_si && d_offsets && d_row_ptr && d_col && d_draws && d_rows && n >= 0 && window >= 0,
                "sgns_explode: bad arguments");
    if (n == 0) return DRB_OK;
    sgns_explode_kernel<<<grid_size(n, 256), 256, 0, (cudaStream_t)stream>>>(d_su, d_si, n, window, d_offsets, d_row_ptr,
                                                                             d_col, d_draws, d_rows);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_mt19937_seed(uint32_t *st, uint32_t seed)
{
    DRB_REQUIRE(st != nullptr, "mt19937_seed: null state");
    for (uint32_t pos = 0; pos < 624; ++pos) {  // init_genrand (numpy _legacy_seeding for an int seed)
        st[pos] = seed;
        seed = 1812433253u * (seed ^ (seed >> 30)) + pos + 1u;
    }
    st[624] = 624;
    return DRB_OK;
}

extern "C" int drb_sampler_draw_mt19937(uint32_t *st, const int64_t *h_row_ptr, int32_t U, int32_t I, int32_t G,
                                        int32_t *h_draws, int32_t *bad_user)
{
    DRB_REQUIRE(st && h_row_ptr && h_draws && U >= 0 && I > 0 && G > 0, "sampler_draw_mt19937: bad arguments");
    Mt mt{st, st + 624};
    for (int32_t u = 0; u < U; ++u) {
        int64_t n = (int64_t)I - (h_row_ptr[u + 1] - h_row_ptr[u]);
        if (n <= 0) {
            if (bad_user) *bad_user = u;
            set_error("'a' cannot be empty: user %d has interacted with every item", u);
            return DRB_ERR_EMPTY_SET;
        }
        for (int32_t g = 0; g < G; ++g) h_draws[(int64_t)u * G + g] = (int32_t)mt.bounded((uint32_t)n);
    }
    return DRB_OK;
}

extern "C" int drb_sampler_draw_mt19937_mixed(uint32_t *st, const int64_t *h_row_ptr, int32_t U, int32_t I,
                                              int32_t uniform_num, int32_t other_num, int32_t *h_draws, double *h_u01,
                                              int32_t *bad_user)
{
    DRB_REQUIRE(st && h_row_ptr && U >= 0 && I > 0 && uniform_num >= 0 && other_num >= 0 && uniform_num + other_num > 0,
                "sampler_draw_mt19937_mixed: bad arguments");
    DRB_REQUIRE((uniform_num == 0 || h_draws) && (other_num == 0 || h_u01), "sampler_draw_mt19937_mixed: null output");
    Mt mt{st, st + 624};
    for (int32_t u = 0; u < U; ++u) {  // per user: uniform ranks first, then the weighted draws (sampler.py:71-80)
        int64_t n = (int64_t)I - (h_row_ptr[u + 1] - h_row_ptr[u]);
        if (n <= 0 && uniform_num > 0) {
            if (bad_user) *bad_user = u;
            set_error("'a' cannot be empty: user %d has interacted with every item", u);
            return DRB_ERR_EMPTY_SET;
        }
        for (int32_t g = 0; g < uniform_num; ++g) h_draws[(int64_t)u * uniform_num + g] = (int32_t)mt.bounded((uint32_t)n);
        for (int32_t g = 0; g < other_num; ++g) h_u01[(int64_t)u * other_num + g] = mt.uniform01();
    }
    return DRB_OK;
}

extern "C" int drb_sampler_assemble_mixed(const int64_t *d_row_ptr, const int32_t *d_col, const int32_t *d_draws,
                                          const double *d_cdf, const double *d_u01, int32_t U, int32_t I,
                                          int32_t uniform_num, int32_t other_num, int32_t *d_js, void *stream)
{
    DRB_REQUIRE(d_row_ptr && d_js && U > 0 && I > 0 && uniform_num >= 0 && other_num >= 0 && uniform_num + other_num > 0,
                "sampler_assemble_mixed: bad arguments");
    DRB_REQUIRE((uniform_num == 0 || d_draws) && (other_num == 0 || (d_cdf && d_u01)), "sampler_assemble_mixed: null input");
    assemble_mixed_kernel<<<grid_size((long long)U * (uniform_num + other_num), 256), 256, 0, (cudaStream_t)stream>>>(
        d_row_ptr, d_col, d_draws, d_cdf, d_u01, U, I, uniform_num, other_num, d_js);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_sampler_explode_pointwise(const int32_t *d_coo_u, const int32_t *d_coo_i, const int32_t *d_label,
                                             int64_t nnz, const int32_t *d_js, int32_t G, int32_t *d_rows, void *stream)
{
    DRB_REQUIRE(d_coo_u && d_coo_i && d_label && d_rows && nnz >= 0 && G >= 0 && (G == 0 || d_js),
                "sampler_explode_pointwise: bad arguments");
    if (nnz == 0) return DRB_OK;
    explode_pointwise_kernel<<<grid_size(nnz * (1 + G), 256), 256, 0, (cudaStream_t)stream>>>(d_coo_u, d_coo_i, d_label,
                                                                                              nnz, d_js, G, d_rows);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_bounded_draws_mt19937(uint32_t *st, const int64_t *h_n, const int64_t *h_offsets, int64_t rows,
                                         int32_t *h_draws, int64_t *bad_row)
{
    DRB_REQUIRE(st && h_n && h_offsets && h_draws && rows >= 0, "bounded_draws_mt19937: bad arguments");
    Mt mt{st, st + 624};
    for (int64_t m = 0; m < rows; ++m) {
        if (h_offsets[m + 1] > h_offsets[m] && h_n[m] <= 0) {
            if (bad_row) *bad_row = m;
            set_error("'a' cannot be empty: row %lld has an empty population", (long long)m);
            return DRB_ERR_EMPTY_SET;
        }
        for (int64_t d = h_offsets[m]; d < h_offsets[m + 1]; ++d) h_draws[d] = (int32_t)mt.bounded((uint32_t)h_n[m]);
    }
    return DRB_OK;
}

extern "C" int drb_kth_complement_var(const int64_t *d_row_ptr, const int32_t *d_col, const int64_t *d_offsets,
                                      const int32_t *d_draws, int64_t rows, int32_t *d_out, void *stream)
{
    DRB_REQUIRE(d_row_ptr && d_offsets && d_draws && d_out && rows >= 0, "kth_complement_var: bad arguments");
    if (rows == 0) return DRB_OK;
    kth_complement_var_kernel<<<grid_size(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(d_row_ptr, d_col, d_offsets,
                                                                                           d_draws, rows, d_out);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_sampler_draw_philox(uint64_t seed, uint64_t offset, const int64_t *d_row_ptr, int32_t U, int32_t I,
                                       int32_t G, int32_t *d_draws, int32_t *d_bad_user, void *stream)
{
    DRB_REQUIRE(d_row_ptr && d_draws && d_bad_user && U > 0 && I > 0 && G > 0, "sampler_draw_philox: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    DRB_CUDA(cudaMemsetAsync(d_bad_user, 0x7f, sizeof(int32_t), st));
    draw_philox_kernel<<<grid_size((long long)U * G, 256), 256, 0, st>>>(seed, offset, d_row_ptr, U, I, G, d_draws,
                                                                         d_bad_user);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_sampler_kth_complement(const int64_t *d_row_ptr, const int32_t *d_col, const int32_t *d_draws,
                                          int32_t U, int32_t I, int32_t G, int32_t *d_js, void *stream)
{
    DRB_REQUIRE(d_row_ptr && d_draws && d_js && U > 0 && I > 0 && G > 0, "sampler_kth_complement: bad arguments");
    kth_complement_kernel<<<grid_size((long long)U * G, 256), 256, 0, (cudaStream_t)stream>>>(d_row_ptr, d_col, d_draws, U,
                                                                                              G, d_js);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_sampler_explode(const int32_t *d_coo_u, const int32_t *d_coo_i, int64_t nnz, const int32_t *d_js,
                                   int32_t G, int32_t *d_triples, void *stream)
{
    DRB_REQUIRE(d_coo_u && d_coo_i && d_js && d_triples && nnz >= 0 && G > 0, "sampler_explode: bad arguments");
    if (nnz == 0) return DRB_OK;
    explode_kernel<<<grid_size(nnz * G, 256), 256, 0, (cudaStream_t)stream>>>(d_coo_u, d_coo_i, nnz, d_js, G, d_triples);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

extern "C" int drb_sample_triples_host(uint32_t *st, const int64_t *h_row_ptr, const int32_t *h_col,
                                       const int32_t *h_coo_u, const int32_t *h_coo_i, int64_t nnz, int32_t U, int32_t I,
                                       int32_t G, int32_t *h_js, int32_t *h_triples, int32_t *bad_user)
{
    DRB_REQUIRE(st && h_row_ptr && h_coo_u && h_coo_i && h_js && h_triples, "sample_triples_host: null argument");
    int32_t *h_draws = h_js;  // draws are overwritten in place by the js table after the device pass
    int rc = drb_sampler_draw_mt19937(st, h_row_ptr, U, I, G, h_draws, bad_user);
    if (rc != DRB_OK) return rc;
    int64_t csr_nnz = h_row_ptr[U];
    int64_t *d_row_ptr = nullptr;
    int32_t *d_col = nullptr, *d_draws = nullptr, *d_js = nullptr, *d_u = nullptr, *d_i = nullptr, *d_tr = nullptr;
    cudaError_t e = cudaSuccess;
    auto A = [&](void **p, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(p, bytes ? bytes : 16);
    };
    A((void **)&d_row_ptr, sizeof(int64_t) * (size_t)(U + 1));
    A((void **)&d_col, sizeof(int32_t) * (size_t)csr_nnz);
    A((void **)&d_draws, sizeof(int32_t) * (size_t)U * G);
    A((void **)&d_js, sizeof(int32_t) * (size_t)U * G);
    A((void **)&d_u, sizeof(int32_t) * (size_t)nnz);
    A((void **)&d_i, sizeof(int32_t) * (size_t)nnz);
    A((void **)&d_tr, sizeof(int32_t) * (size_t)nnz * G * 3);
    auto C = [&](void *d, const void *h, size_t bytes, cudaMemcpyKind k) {
        if (e == cudaSuccess && bytes) e = cudaMemcpy(d, h, bytes, k);
    };
    C(d_row_ptr, h_row_ptr, sizeof(int64_t) * (size_t)(U + 1), cudaMemcpyHostToDevice);
    C(d_col, h_col, sizeof(int32_t) * (size_t)csr_nnz, cudaMemcpyHostToDevice);
    C(d_draws, h_draws, sizeof(int32_t) * (size_t)U * G, cudaMemcpyHostToDevice);
    C(d_u, h_coo_u, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice);
    C(d_i, h_coo_i, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = drb_sampler_kth_complement(d_row_ptr, d_col, d_draws, U, I, G, d_js, nullptr);
        if (rc == DRB_OK) rc = drb_sampler_explode(d_u, d_i, nnz, d_js, G, d_tr, nullptr);
        if (rc == DRB_OK) e = cudaDeviceSynchronize();
    }
    C(h_js, d_js, sizeof(int32_t) * (size_t)U * G, cudaMemcpyDeviceToHost);
    C(h_triples, d_tr, sizeof(int32_t) * (size_t)nnz * G * 3, cudaMemcpyDeviceToHost);
    cudaFree(d_row_ptr); cudaFree(d_col); cudaFree(d_draws); cudaFree(d_js); cudaFree(d_u); cudaFree(d_i); cudaFree(d_tr);
    if (e != cudaSuccess) return cuda_fail(e, "sample_triples_host", __FILE__, __LINE__);
    return rc;
}
