// csr.cu -- host-side producers of the hot path's inputs, rebuilt on the device.
//
// The reference derives every structure the pair-wise path consumes from the train DataFrame with Python
// loops: get_ur (daisy/utils/utils.py:19-34, iterrows into dict-of-sets), the sampler's per-user
// setdiff1d (daisy/utils/sampler.py:84-89), get_inter_matrix (utils.py:125-144) and LightGCN's
// get_norm_adj_mat (daisy/model/LightGCNRecommender.py:73-107: dok_matrix updates + D^-1/2 A D^-1/2 in
// scipy).  All of them are views of ONE object: the interaction set as a sorted, duplicate-free CSR.
//
//   drb_csr_build        COO (row, col) pairs in any order, duplicates allowed  ->  CSR with ascending,
//                        unique columns per row (set semantics of get_ur / dok_matrix):
//                          count -> scan -> scatter (groups a row's entries, unordered)
//                          -> per row: mark a bitmap of n_cols bits in shared memory (sorts AND removes
//                             duplicates in one step), popcount -> scan -> re-mark and emit in order.
//                        O(nnz + n_rows * n_cols / 32) word operations, no comparison sort.
//   drb_lgcn_build_adj   the user->item CSR and its transpose  ->  A_hat of get_norm_adj_mat as CSR over
//                        the U+I nodes: row r < U lists U + item, row U + i lists users;
//                        val = float32(d_r * d_c), d = (deg + 1e-7)^-1/2 in fp64 like scipy's
//                        (D * A * D).  The reciprocal square root is 1/sqrt (IEEE) where numpy calls pow:
//                        results agree to the last fp32 bit except on rare rounding ties (tested: 1 ulp).
#include "common.cuh"

namespace drb {

constexpr int kCsrThreads = 128;
constexpr int kCsrMaxCols = 1 << 20;  // bitmap of n_cols bits must fit shared memory (128 KiB)

__global__ void csr_count_kernel(const int32_t *__restrict__ row, long long nnz, int n_rows, unsigned *__restrict__ deg,
                                 int *__restrict__ bad)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (long long)gridDim.x * blockDim.x) {
        int r = __ldg(row + k);
        if (r < 0 || r >= n_rows) { *bad = 1; continue; }
        atomicAdd(deg + r, 1u);
    }
}

// exclusive scan of n counters into int64 offsets, out[n] = total.  One CTA: n is a row count (<= a few 10^5).
__global__ void __launch_bounds__(1024) csr_exscan_kernel(const unsigned *__restrict__ in, int64_t *__restrict__ out, long long n)
{
    __shared__ long long wtot[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long carry = 0;
    for (long long base = 0; base < n; base += 1024) {
        const long long idx = base + tid;
        const long long v = idx < n ? (long long)in[idx] : 0;
        long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            long long y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wtot[warp] = x;
        __syncthreads();
        if (warp == 0) {
            long long t = wtot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                long long y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            wtot[lane] = t;
        }
        __syncthreads();
        if (idx < n) out[idx] = carry + (warp > 0 ? wtot[warp - 1] : 0) + x - v;
        const long long total = wtot[31];
        __syncthreads();
        carry += total;
    }
    if (tid == 0) out[n] = carry;
}

__global__ void csr_scatter_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col, long long nnz,
                                   int n_rows, int n_cols, const int64_t *__restrict__ raw_ptr, unsigned *__restrict__ cursor,
                                   int32_t *__restrict__ tmp, int *__restrict__ bad)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (long long)gridDim.x * blockDim.x) {
        int r = __ldg(row + k), c = __ldg(col + k);
        if (r < 0 || r >= n_rows) continue;
        if (c < 0 || c >= n_cols) { *bad = 1; c = 0; }
        tmp[raw_ptr[r] + atomicAdd(cursor + r, 1u)] = c;
    }
}

// One CTA per row (grid-stride).  EMIT = false: uniq[r] = number of distinct columns.  EMIT = true: write them,
// ascending, at out[ptr[r] ...].
template <bool EMIT>
__global__ void __launch_bounds__(kCsrThreads) csr_rows_kernel(const int64_t *__restrict__ raw_ptr, const int32_t *__restrict__ tmp,
                                                              int n_rows, int n_cols, unsigned *__restrict__ uniq,
                                                              const int64_t *__restrict__ ptr, int32_t *__restrict__ out)
{
    extern __shared__ uint32_t bits[];
    __shared__ int wsum[kCsrThreads / 32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int words = (n_cols + 31) >> 5;
    for (int r = blockIdx.x; r < n_rows; r += gridDim.x) {
        const long long b = raw_ptr[r], e = raw_ptr[r + 1];
        if (e == b) {
            if (!EMIT && tid == 0) uniq[r] = 0u;
            continue;  // uniform across the CTA
        }
        for (int w = tid; w < words; w += kCsrThreads) bits[w] = 0u;
        __syncthreads();
        for (long long k = b + tid; k < e; k += kCsrThreads) {
            const int c = __ldg(tmp + k);
            atomicOr(&bits[c >> 5], 1u << (c & 31));
        }
        __syncthreads();
        if (tid == 0) s_base = 0;
        __syncthreads();
        for (int w0 = 0; w0 < words; w0 += kCsrThreads) {
            const int w = w0 + tid;
            const uint32_t m = w < words ? bits[w] : 0u;
            const int pc = __popc(m);
            int x = pc;  // inclusive scan over the CTA
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            if (lane == 31) wsum[warp] = x;
            __syncthreads();
            int before = s_base;
            for (int q = 0; q < warp; ++q) before += wsum[q];
            if (EMIT) {
                long long o = ptr[r] + before + (x - pc);
                uint32_t mm = m;
                while (mm) {
                    const int bit = __ffs(mm) - 1;
                    mm &= mm - 1;
                    out[o++] = w * 32 + bit;
                }
            }
            __syncthreads();
            if (tid == kCsrThreads - 1) s_base = before + x;
            __syncthreads();
        }
        if (!EMIT && tid == 0) uniq[r] = (unsigned)s_base;
        __syncthreads();
    }
}

// A_hat rows: r < U -> (U + item, d_r d_c); r >= U -> (user, d_r d_c).  One thread per stored entry.
__global__ void lgcn_adj_kernel(const int64_t *__restrict__ ui_ptr, const int32_t *__restrict__ ui_col,
                                const int64_t *__restrict__ iu_ptr, const int32_t *__restrict__ iu_col, int U, int I,
                                long long nnz, int64_t *__restrict__ adj_ptr, int32_t *__restrict__ adj_col,
                                float *__restrict__ adj_val)
{
    const long long total = 2 * nnz, nodes = (long long)U + I;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total + nodes + 1;
         k += (long long)gridDim.x * blockDim.x) {
        if (k >= total) {  // the row pointer
            const long long r = k - total;
            adj_ptr[r] = r <= U ? ui_ptr[r < U ? r : U] : nnz + iu_ptr[r - U];
            continue;
        }
        const bool urow = k < nnz;
        const int64_t *ptr = urow ? ui_ptr : iu_ptr;
        const long long pos = urow ? k : k - nnz;
        const int n = urow ? U : I;
        int lo = 0, hi = n;  // row of entry pos: last r with ptr[r] <= pos
        while (hi - lo > 1) {
            int mid = (lo + hi) >> 1;
            if (ptr[mid] <= pos) lo = mid; else hi = mid;
        }
        const int c = urow ? __ldg(ui_col + pos) : __ldg(iu_col + pos);
        const double dr = (double)(ptr[lo + 1] - ptr[lo]) + 1e-7;
        const int64_t *optr = urow ? iu_ptr : ui_ptr;
        const double dc = (double)(optr[c + 1] - optr[c]) + 1e-7;
        adj_col[k] = urow ? U + c : c;
        adj_val[k] = (float)((1.0 / sqrt(dr)) * (1.0 / sqrt(dc)));
    }
}

struct CsrWs {
    unsigned *deg, *cursor, *uniq;
    int64_t *raw_ptr;
    int32_t *tmp;
    int *bad;
};

static size_t carve_csr(void *base, int n_rows, long long nnz, CsrWs *w)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) {
        char *p = b ? b + off : nullptr;
        off += (bytes + 255) & ~(size_t)255;
        return p;
    };
    CsrWs t;
    t.bad = (int *)take(256);
    t.deg = (unsigned *)take(sizeof(unsigned) * (size_t)n_rows);
    t.cursor = (unsigned *)take(sizeof(unsigned) * (size_t)n_rows);
    t.uniq = (unsigned *)take(sizeof(unsigned) * (size_t)n_rows);
    t.raw_ptr = (int64_t *)take(sizeof(int64_t) * ((size_t)n_rows + 1));
    t.tmp = (int32_t *)take(sizeof(int32_t) * (size_t)(nnz > 0 ? nnz : 1));
    if (w) *w = t;
    return off;
}

}  // namespace drb

using namespace drb;

extern "C" size_t drb_csr_workspace_bytes(int32_t n_rows, int64_t nnz)
{
    if (n_rows <= 0 || nnz < 0) return 0;
    return carve_csr(nullptr, n_rows, nnz, nullptr);
}

extern "C" int drb_csr_build(const int32_t *d_row, const int32_t *d_col, int64_t nnz, int32_t n_rows, int32_t n_cols,
                             void *d_ws, int64_t *d_row_ptr, int32_t *d_col_out, int64_t *h_nnz_unique, void *stream)
{
    DRB_REQUIRE(d_ws && d_row_ptr && d_col_out && nnz >= 0 && n_rows > 0 && n_cols > 0 && (nnz == 0 || (d_row && d_col)),
                "csr_build: bad arguments");
    DRB_REQUIRE(n_cols <= kCsrMaxCols, "csr_build: n_cols %d exceeds the %d-bit row bitmap", n_cols, kCsrMaxCols);
    cudaStream_t st = (cudaStream_t)stream;
    CsrWs w;
    carve_csr(d_ws, n_rows, nnz, &w);
    // bad flag, deg, cursor are contiguous at the start of the workspace: one memset
    DRB_CUDA(cudaMemsetAsync(d_ws, 0, (size_t)((char *)w.uniq - (char *)d_ws), st));
    if (nnz) csr_count_kernel<<<grid_size(nnz, 256), 256, 0, st>>>(d_row, nnz, n_rows, w.deg, w.bad);
    csr_exscan_kernel<<<1, 1024, 0, st>>>(w.deg, w.raw_ptr, n_rows);
    if (nnz) csr_scatter_kernel<<<grid_size(nnz, 256), 256, 0, st>>>(d_row, d_col, nnz, n_rows, n_cols, w.raw_ptr, w.cursor, w.tmp, w.bad);
    const size_t smem = sizeof(uint32_t) * (size_t)((n_cols + 31) / 32);
    if (smem > 48 * 1024) {
        DRB_CUDA(cudaFuncSetAttribute(csr_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DRB_CUDA(cudaFuncSetAttribute(csr_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    long long cap = (long long)sm_count() * (smem > 32 * 1024 ? 2 : 8);
    const int grid = (int)(n_rows < cap ? n_rows : cap);
    csr_rows_kernel<false><<<grid, kCsrThreads, smem, st>>>(w.raw_ptr, w.tmp, n_rows, n_cols, w.uniq, nullptr, nullptr);
    csr_exscan_kernel<<<1, 1024, 0, st>>>(w.uniq, d_row_ptr, n_rows);
    csr_rows_kernel<true><<<grid, kCsrThreads, smem, st>>>(w.raw_ptr, w.tmp, n_rows, n_cols, nullptr, d_row_ptr, d_col_out);
    DRB_CUDA(cudaGetLastError());
    int bad = 0;
    int64_t total = 0;
    DRB_CUDA(cudaMemcpyAsync(&bad, w.bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    DRB_CUDA(cudaMemcpyAsync(&total, d_row_ptr + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    DRB_CUDA(cudaStreamSynchronize(st));
    DRB_REQUIRE(bad == 0, "csr_build: an index lies outside [0, %d) x [0, %d)", n_rows, n_cols);
    if (h_nnz_unique) *h_nnz_unique = total;
    return DRB_OK;
}

extern "C" int drb_lgcn_build_adj(const int64_t *d_ui_ptr, const int32_t *d_ui_col, const int64_t *d_iu_ptr,
                                  const int32_t *d_iu_col, int32_t U, int32_t I, int64_t nnz, int64_t *d_adj_ptr,
                                  int32_t *d_adj_col, float *d_adj_val, void *stream)
{
    DRB_REQUIRE(d_ui_ptr && d_iu_ptr && d_adj_ptr && U > 0 && I > 0 && nnz >= 0, "lgcn_build_adj: bad arguments");
    DRB_REQUIRE(nnz == 0 || (d_ui_col && d_iu_col && d_adj_col && d_adj_val), "lgcn_build_adj: null arrays");
    lgcn_adj_kernel<<<grid_size(2 * nnz + U + I + 1, 256), 256, 0, (cudaStream_t)stream>>>(d_ui_ptr, d_ui_col, d_iu_ptr, d_iu_col, U, I,
                                                                                           nnz, d_adj_ptr, d_adj_col, d_adj_val);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}
