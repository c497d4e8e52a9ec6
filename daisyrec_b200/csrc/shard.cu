// shard.cu -- train feed for user-sharded multi-GPU training (SURVEY 8(e)).
//
// Every rank walks the SAME global epoch permutation (daisy/utils/dataset.py:5-27 semantics) and
// keeps the triples whose user it owns, so the union of the ranks' local batches of step s is
// exactly the single-GPU batch s.  Three passes over the permutation:
//   count   : owned triples per global step            (one atomic per owned triple)
//   scan    : exclusive prefix over the steps           (single CTA; n_steps+1 entries)
//   scatter : write local-user-id SoA planes at offsets[s] + cursor[s]++  (order inside a step is
//             irrelevant: a step is a sum over its batch)
#include "common.cuh"

namespace drb {

__global__ void shard_count_kernel(const int32_t *__restrict__ triples, const int64_t *__restrict__ perm, long long n,
                                   int user_lo, int user_hi, long long batch, unsigned long long *__restrict__ counts)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        long long src = perm ? perm[k] : k;
        int u = __ldg(triples + 3 * src);
        if (u >= user_lo && u < user_hi) atomicAdd(counts + k / batch, 1ull);
    }
}

// offsets[0..m] = exclusive scan of counts[0..m); counts[] is reused as the scatter cursors (zeroed)
__global__ void shard_scan_kernel(unsigned long long *__restrict__ counts, long long m, long long *__restrict__ offsets)
{
    __shared__ unsigned long long s_part[1024];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (long long base = 0; base < m; base += blockDim.x) {
        long long i = base + threadIdx.x;
        unsigned long long v = i < m ? counts[i] : 0;
        s_part[threadIdx.x] = v;
        __syncthreads();
        for (int off = 1; off < blockDim.x; off <<= 1) {      // Hillis-Steele inclusive scan
            unsigned long long t = threadIdx.x >= off ? s_part[threadIdx.x - off] : 0;
            __syncthreads();
            s_part[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < m) {
            offsets[i] = (long long)(s_carry + s_part[threadIdx.x] - v);
            counts[i] = 0;
        }
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry += s_part[threadIdx.x];
        __syncthreads();
    }
    if (threadIdx.x == 0) offsets[m] = (long long)s_carry;
}

__global__ void shard_scatter_kernel(const int32_t *__restrict__ triples, const int64_t *__restrict__ perm, long long n,
                                     int user_lo, int user_hi, long long batch, const long long *__restrict__ offsets,
                                     unsigned long long *__restrict__ cursors, int32_t *__restrict__ bu,
                                     int32_t *__restrict__ bi, int32_t *__restrict__ bj)
{
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        long long src = perm ? perm[k] : k;
        const int32_t *t = triples + 3 * src;
        int u = __ldg(t);
        if (u >= user_lo && u < user_hi) {
            long long s = k / batch;
            long long pos = offsets[s] + (long long)atomicAdd(cursors + s, 1ull);
            bu[pos] = u - user_lo;
            bi[pos] = __ldg(t + 1);
            bj[pos] = __ldg(t + 2);
        }
    }
}

}  // namespace drb

using namespace drb;

extern "C" int drb_shard_gather_triples(const int32_t *d_triples, const int64_t *d_perm, int64_t n, int32_t user_lo,
                                        int32_t user_hi, int64_t batch, unsigned long long *d_scratch_counts,
                                        int64_t *d_step_offsets, int32_t *d_bu, int32_t *d_bi, int32_t *d_bj,
                                        void *stream)
{
    DRB_REQUIRE(d_triples && d_scratch_counts && d_step_offsets && d_bu && d_bi && d_bj && n >= 0 && batch > 0 &&
                    user_lo <= user_hi,
                "shard_gather_triples: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    long long m = (n + batch - 1) / batch;
    DRB_CUDA(cudaMemsetAsync(d_scratch_counts, 0, sizeof(unsigned long long) * (size_t)(m > 0 ? m : 1), st));
    if (n > 0) {
        const int blocks = grid_size(n, 256);
        shard_count_kernel<<<blocks, 256, 0, st>>>(d_triples, d_perm, n, user_lo, user_hi, batch, d_scratch_counts);
        shard_scan_kernel<<<1, 1024, 0, st>>>(d_scratch_counts, m, (long long *)d_step_offsets);
        shard_scatter_kernel<<<blocks, 256, 0, st>>>(d_triples, d_perm, n, user_lo, user_hi, batch,
                                                     (const long long *)d_step_offsets, d_scratch_counts, d_bu, d_bi, d_bj);
    } else {
        DRB_CUDA(cudaMemsetAsync(d_step_offsets, 0, sizeof(int64_t), st));
    }
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}
