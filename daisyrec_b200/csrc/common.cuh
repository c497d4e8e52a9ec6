// common.cuh -- shared device/host helpers of libdaisyrec_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/daisyrec_b200.h"

namespace drb {

// ---------------------------------------------------------------- host-side error plumbing
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define DRB_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t _e = (call);                                                    \
        if (_e != cudaSuccess) return drb::cuda_fail(_e, #call, __FILE__, __LINE__); \
    } while (0)

#define DRB_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            drb::set_error(__VA_ARGS__);  \
            return DRB_ERR_INVALID;       \
        }                                 \
    } while (0)

int sm_count();

// blocks of a grid-stride loop over n items: one per `block` items, at most per_sm per SM, at least one
inline int grid_size(long long n, int block, int per_sm = 16)
{
    long long b = (n + block - 1) / block, cap = (long long)sm_count() * per_sm;
    if (b > cap) b = cap;
    return (int)(b < 1 ? 1 : b);
}

// ---------------------------------------------------------------- row geometry
// A factor row of F floats is processed by a group of W lanes (W a power of two <= 32);
// lane l owns the chunks c = l, l+W, ... of VEC consecutive floats (NCH chunks per lane at most).
// This fixes the canonical fp32 summation order of every dot product (DESIGN.md, oracle orc_dot).
struct RowGeom {
    int vec, width, nch;
};
inline RowGeom row_geom(int F)
{
    RowGeom g;
    g.vec = (F % 4 == 0) ? 4 : (F % 2 == 0) ? 2 : 1;
    int chunks = F / g.vec;
    g.width = 1;
    while (g.width < chunks && g.width < 32) g.width <<= 1;
    int per = (chunks + g.width - 1) / g.width;
    g.nch = 1;
    while (g.nch < per) g.nch <<= 1;
    return g;
}

#ifdef __CUDACC__
// ---------------------------------------------------------------- vector row access
template <int VEC>
struct Vec;
template <>
struct Vec<4> {
    float v[4];
};
template <>
struct Vec<2> {
    float v[2];
};
template <>
struct Vec<1> {
    float v[1];
};

// L2-coherent (ld.global.cg) loads: tables are updated by other SMs between the phases of the
// persistent kernel, so rows must never be served from a stale L1 line.
template <int VEC>
__device__ __forceinline__ Vec<VEC> ld_row(const float *p)
{
    Vec<VEC> r;
    if constexpr (VEC == 4) {
        float4 t = __ldcg(reinterpret_cast<const float4 *>(p));
        r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
    } else if constexpr (VEC == 2) {
        float2 t = __ldcg(reinterpret_cast<const float2 *>(p));
        r.v[0] = t.x; r.v[1] = t.y;
    } else {
        r.v[0] = __ldcg(p);
    }
    return r;
}

template <int VEC>
__device__ __forceinline__ void st_row(float *p, const Vec<VEC> &r)
{
    if constexpr (VEC == 4) {
        __stcg(reinterpret_cast<float4 *>(p), make_float4(r.v[0], r.v[1], r.v[2], r.v[3]));
    } else if constexpr (VEC == 2) {
        __stcg(reinterpret_cast<float2 *>(p), make_float2(r.v[0], r.v[1]));
    } else {
        __stcg(p, r.v[0]);
    }
}

// Fire-and-forget vector reduction into L2 (RED.E.ADD.F32x4 on sm_90+): one instruction
// adds VEC consecutive floats, no return value, no L1 involvement.
template <int VEC>
__device__ __forceinline__ void red_row(float *p, const Vec<VEC> &r)
{
    if constexpr (VEC == 4) {
        asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]),
                     "f"(r.v[2]), "f"(r.v[3])
                     : "memory");
    } else if constexpr (VEC == 2) {
        asm volatile("red.relaxed.gpu.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]) : "memory");
    } else {
        asm volatile("red.relaxed.gpu.global.add.f32 [%0], %1;" ::"l"(p), "f"(r.v[0]) : "memory");
    }
}

__device__ __forceinline__ void red_add_u32(unsigned *p, unsigned v)
{
    asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_add_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// xor-butterfly sum over the W lanes of a group (W consecutive lanes, W | 32)
template <int W>
__device__ __forceinline__ float group_sum(float x)
{
#pragma unroll
    for (int off = W >> 1; off >= 1; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

__device__ __forceinline__ double warp_sum(double x)
{
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

// ---------------------------------------------------------------- factor rows in registers
template <int VEC, int W, int NCH>
struct Row {
    Vec<VEC> c[NCH];
};

template <int VEC, int W, int NCH>
__device__ __forceinline__ Row<VEC, W, NCH> load_row(const float *base, int gl, int chunks, bool valid)
{
    Row<VEC, W, NCH> r;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        int c = gl + ch * W;
        if (valid && c < chunks) {
            r.c[ch] = ld_row<VEC>(base + c * VEC);
        } else {
#pragma unroll
            for (int e = 0; e < VEC; ++e) r.c[ch].v[e] = 0.f;
        }
    }
    return r;
}

// canonical dot: per-lane sequential fmaf over its chunks, then xor-butterfly over the W lanes
template <int VEC, int W, int NCH>
__device__ __forceinline__ float dot_rows(const Row<VEC, W, NCH> &a, const Row<VEC, W, NCH> &b)
{
    float acc = 0.f;
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
        for (int e = 0; e < VEC; ++e) acc = fmaf(a.c[ch].v[e], b.c[ch].v[e], acc);
    return group_sum<W>(acc);
}

// ---------------------------------------------------------------- mbarrier + 1-D bulk TMA
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// cp.async.bulk (UBLKCP): contiguous global -> shared copy performed by the TMA unit;
// src, dst 16-byte aligned, bytes a multiple of 16; completion counted on the mbarrier.
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- Philox4x32-10 (device)
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1)
{
    uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
__device__ __forceinline__ void philox4x32(uint32_t (&c)[4], uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

// ---------------------------------------------------------------- grid-wide barrier
// All CTAs of a cooperative launch are co-resident.  Monotonic ticket barrier: the counter is
// zeroed by the host before the launch; barrier number k completes when it reaches k*gridDim.x.
__device__ __forceinline__ void grid_barrier(unsigned long long *counter, unsigned long long &epoch)
{
    __syncthreads();
    epoch += gridDim.x;
    if (threadIdx.x == 0) {
        __threadfence();                       // publish this CTA's writes / reductions
        atomicAdd(counter, 1ull);
        unsigned long long seen;
        do {
            asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(counter) : "memory");
        } while (seen < epoch);
    }
    __syncthreads();
}
#endif  // __CUDACC__

}  // namespace drb
