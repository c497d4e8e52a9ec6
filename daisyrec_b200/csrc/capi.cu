// capi.cu -- library-level entry points and error plumbing of libdaisyrec_b200.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace drb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    set_error("CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file, line);
    cudaGetLastError();  // clear the sticky-less error state
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorNoKernelImageForDevice ||
        e == cudaErrorInvalidDeviceFunction)
        return DRB_ERR_NO_DEVICE;
    return DRB_ERR_CUDA;
}

int sm_count()
{
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return 148;
        cached = prop.multiProcessorCount;
        cached_dev = dev;
    }
    return cached;
}

// out[c] += number of ids of column c outside [0, hi[c]); ids laid out [n, ncols] row-major (ncols <= 4)
template <typename T>
__global__ void index_range_kernel(const T *__restrict__ ids, long long n, int ncols, const long long *__restrict__ hi4,
                                   unsigned long long *__restrict__ out4)
{
    unsigned long long bad[4] = {0, 0, 0, 0};
    const long long total = n * ncols;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(k % ncols);
        const long long v = (long long)ids[k];
        if (v < 0 || v >= hi4[c]) ++bad[c];
    }
    for (int c = 0; c < ncols; ++c) {
        unsigned long long v = bad[c];
        for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(out4 + c, v);
    }
}

}  // namespace drb

extern "C" int drb_version(void) { return 202; }

// nn.Embedding raises IndexError for an id outside its table (torch/nn/functional.py embedding); the kernels index raw
// tables, so fit() / rank() run this check once per uploaded index array.  h_bad[c] = ids of column c outside [0, h_hi[c]).
extern "C" int drb_index_range_check(const void *d_ids, int32_t elem_bytes, int64_t n_rows, int32_t n_cols,
                                     const int64_t *h_hi, int64_t *h_bad, void *stream)
{
    using namespace drb;
    DRB_REQUIRE(d_ids && h_hi && h_bad && n_rows >= 0 && n_cols >= 1 && n_cols <= 4 && (elem_bytes == 4 || elem_bytes == 8),
                "index_range_check: bad arguments");
    for (int c = 0; c < n_cols; ++c) h_bad[c] = 0;
    if (n_rows == 0) return DRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local long long *d_buf = nullptr;     // [0..3] bounds, [4..7] counters
    if (!d_buf) DRB_CUDA(cudaMalloc(&d_buf, 8 * sizeof(long long)));
    long long h_buf[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int c = 0; c < n_cols; ++c) h_buf[c] = h_hi[c];
    DRB_CUDA(cudaMemcpyAsync(d_buf, h_buf, sizeof(h_buf), cudaMemcpyHostToDevice, st));
    long long blocks = (n_rows * n_cols + 1023) / 1024, cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (elem_bytes == 4)
        index_range_kernel<int32_t><<<(int)blocks, 256, 0, st>>>((const int32_t *)d_ids, n_rows, n_cols, d_buf,
                                                                 (unsigned long long *)(d_buf + 4));
    else
        index_range_kernel<int64_t><<<(int)blocks, 256, 0, st>>>((const int64_t *)d_ids, n_rows, n_cols, d_buf,
                                                                 (unsigned long long *)(d_buf + 4));
    DRB_CUDA(cudaGetLastError());
    DRB_CUDA(cudaMemcpyAsync(h_buf, d_buf, sizeof(h_buf), cudaMemcpyDeviceToHost, st));
    DRB_CUDA(cudaStreamSynchronize(st));
    for (int c = 0; c < n_cols; ++c) h_bad[c] = h_buf[4 + c];
    return DRB_OK;
}

extern "C" const char *drb_last_error(void) { return drb::g_err; }

extern "C" int drb_device_query(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor, int64_t *l2_bytes)
{
    int dev = 0;
    DRB_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    DRB_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (l2_bytes) *l2_bytes = prop.l2CacheSize;
    return DRB_OK;
}
