// Shared device helpers for the sm_100a kernels: mbarrier, TMA, tcgen05/TMEM wrappers (inline PTX), bf16 packing.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

namespace tmae {

// Every kernel of the library asks for the same (maximum) shared-memory carve-out, so the SMs never have to
// reconfigure the L1/shared split between the smem-heavy GEMM launches and the small kernels around them.
template <typename K>
inline void prefer_max_smem_carveout(K kernel) {
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
#define TMAE_CARVEOUT_ONCE(kernel)                       \
    do {                                                 \
        static bool _done = false;                       \
        if (!_done) { prefer_max_smem_carveout(kernel); _done = true; } \
    } while (0)

// --------------------------------------------------------------------------------------------
// small math
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float v) {          // nn.GELU() default (exact erf form)
    return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
// split-bf16 pair of two fp32 values: hi = bf16(v), lo = bf16(v - hi)  (hi + lo carries 16 mantissa bits of v)
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const float2 hf = __bfloat1622float2(h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(a - hf.x, b - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
// Store 4 consecutive bf16 outputs, as 1, 2 or 3 planes.  `lo_off` encodes the plane layout of the destination buffer:
//   0  one plane (plain bf16);  > 0  two planes (hi, lo) `lo_off` elements apart (split-bf16, 16 mantissa bits);
//   < 0  three planes (hi, mid, lo) `-lo_off` elements apart (24 mantissa bits: fp32 carried exactly).
__device__ __forceinline__ void store_bf16x4_planes(__nv_bfloat16* dst, long long lo_off, float v0, float v1, float v2, float v3) {
    if (lo_off == 0) {
        uint2 pk;
        pk.x = pack_bf16x2(v0, v1);
        pk.y = pack_bf16x2(v2, v3);
        *reinterpret_cast<uint2*>(dst) = pk;
        return;
    }
    const long long stride = lo_off > 0 ? lo_off : -lo_off;
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(v0, v1), h1 = __floats2bfloat162_rn(v2, v3);
    const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
    const float r0 = v0 - f0.x, r1 = v1 - f0.y, r2 = v2 - f1.x, r3 = v3 - f1.y;       // exact in fp32
    const __nv_bfloat162 m0 = __floats2bfloat162_rn(r0, r1), m1 = __floats2bfloat162_rn(r2, r3);
    uint2 pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&h0); pk.y = *reinterpret_cast<const uint32_t*>(&h1);
    *reinterpret_cast<uint2*>(dst) = pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&m0); pk.y = *reinterpret_cast<const uint32_t*>(&m1);
    *reinterpret_cast<uint2*>(dst + stride) = pk;
    if (lo_off < 0) {
        const float2 g0 = __bfloat1622float2(m0), g1 = __bfloat1622float2(m1);
        pk.x = pack_bf16x2(r0 - g0.x, r1 - g0.y);
        pk.y = pack_bf16x2(r2 - g1.x, r3 - g1.y);
        *reinterpret_cast<uint2*>(dst + 2 * stride) = pk;
    }
}
// scalar form of the same layout
__device__ __forceinline__ void store_bf16_planes(__nv_bfloat16* dst, long long lo_off, float v) {
    const __nv_bfloat16 h = __float2bfloat16(v);
    dst[0] = h;
    if (lo_off == 0) return;
    const long long stride = lo_off > 0 ? lo_off : -lo_off;
    const float r = v - __bfloat162float(h);
    const __nv_bfloat16 m = __float2bfloat16(r);
    dst[stride] = m;
    if (lo_off < 0) dst[2 * stride] = __float2bfloat16(r - __bfloat162float(m));
}
// sum of the planes of one element (precise attention reads q, k, v this way)
__device__ __forceinline__ float load_bf16_planes(const __nv_bfloat16* src, long long lo_off) {
    float v = __bfloat162float(src[0]);
    if (lo_off == 0) return v;
    const long long stride = lo_off > 0 ? lo_off : -lo_off;
    v += __bfloat162float(src[stride]);
    if (lo_off < 0) v += __bfloat162float(src[2 * stride]);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Gaussian conditional likelihood + quantisation of one element (compressai GaussianConditional eval forward + quantize_ste,
// MCM.py:771-776): shared by gaussian_slice_kernel and the fused epilogue of the cc_transform nets' last layer.
__device__ __forceinline__ void gaussian_elem(float y, float mu, float sigma, float& lik, float& sym, float& yhat) {
    const float kNegInvSqrt2 = -0.70710678118654752440f;        // float(-(2 ** -0.5))
    sym = rintf(y - mu);
    yhat = sym + mu;
    const float d = fabsf(yhat - mu);
    const float s = fmaxf(sigma, 0.11f);
    const float upper = 0.5f * erfcf(kNegInvSqrt2 * ((0.5f - d) / s));
    const float lower = 0.5f * erfcf(kNegInvSqrt2 * ((-0.5f - d) / s));
    lik = fmaxf(upper - lower, 1e-9f);
}

// compressai GaussianConditional.build_indexes (MCM.py:839) of four scales: lower-bounded at 0.11, then
// index = (len - 1) - #{t in table[:-1] : scale <= t}  ==  #{t in table[:-1] : t < scale}.
// The one definition behind every scale-table index the library emits (encoder and decoder must agree bit for bit).
__device__ __forceinline__ int4 scale_indexes4(const float* __restrict__ table, int n_table, float4 sv) {
    const float sc[4] = {fmaxf(sv.x, 0.11f), fmaxf(sv.y, 0.11f), fmaxf(sv.z, 0.11f), fmaxf(sv.w, 0.11f)};
    int id[4] = {0, 0, 0, 0};
    for (int t = 0; t < n_table - 1; ++t) {
        const float tv = __ldg(table + t);
#pragma unroll
        for (int e = 0; e < 4; ++e) id[e] += (tv < sc[e]) ? 1 : 0;
    }
    return make_int4(id[0], id[1], id[2], id[3]);
}

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-stream-serialization attribute may start
// while its predecessor is still running; everything before pdl_wait() (barrier init, TMEM allocation, descriptor
// prefetch) overlaps the predecessor's tail, pdl_wait() blocks until the predecessor has completed and flushed.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

inline bool pdl_enabled() {
    static const bool on = getenv("TMAE_NO_PDL") == nullptr;
    return on;
}
// Launch helper: `pdl` = allow this kernel to overlap the tail of the previous kernel in the stream.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (pdl && pdl_enabled()) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Same with a thread-block cluster of `cluster_x` CTAs along x (CTA pairs for cta_group::2 kernels).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, int cluster_x,
                                    Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster_x; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (pdl && pdl_enabled()) ? 2 : 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

__device__ __forceinline__ long long globaltimer_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// --------------------------------------------------------------------------------------------
// shared-memory addresses, elect
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// --------------------------------------------------------------------------------------------
// mbarrier
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must become a trapped kernel (reported error), never a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {   // ~2 s
            printf("tmae: mbarrier wait timed out (block %d,%d thread %d parity %u)\n", blockIdx.x, blockIdx.y,
                   threadIdx.x, parity);
            __trap();
        }
    }
}

// explicit shared-space vector accesses (a pointer derived from the manually aligned dynamic-smem base is a generic
// pointer to the compiler, which would emit slower generic LD/ST for it)
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// 32-bit shared-address variants for the hot loops (no generic->shared conversion per call)
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// non-blocking probe (try_wait may suspend the thread for a system-dependent time when the phase is not complete)
__device__ __forceinline__ bool mbar_test_wait_a(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait_a(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait_a(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {   // ~2 s
            printf("tmae: mbarrier wait timed out (block %d,%d thread %d parity %u)\n", blockIdx.x, blockIdx.y,
                   threadIdx.x, parity);
            __trap();
        }
    }
}
__device__ __forceinline__ void mbar_arrive_expect_tx_a(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d_a(uint32_t smem_dst, const void* tmap, uint32_t bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
            "r"(smem_dst),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_a(uint32_t smem_dst, const void* tmap, uint32_t bar, int32_t c0, int32_t c1,
                                              int32_t c2, int32_t c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::
            "r"(smem_dst),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// TMA store of a 2-D tile (shared -> global, clipped to the tensor map's bounds), bulk async-group bookkeeping
__device__ __forceinline__ void tma_store_2d_a(const void* tmap, uint32_t smem_src, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n" ::"l"(reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d_a(const void* tmap, uint32_t smem_src, int32_t c0, int32_t c1, int32_t c2, int32_t c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];\n" ::"l"(reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(N) : "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(threads) : "memory"); }
// fire-and-forget L2 prefetch of a global range (16-byte aligned address, size a multiple of 16)
__device__ __forceinline__ void l2_prefetch_bulk(const void* gptr, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(reinterpret_cast<uint64_t>(gptr)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}

// --------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor), 2-D tiles, completion on an mbarrier
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
            "r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// --------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_dst)),
                 "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // whole warp (the allocating one)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
                 : "memory");
}
// 32 lanes x 32 columns of fp32 accumulator -> 32 registers per thread (thread i <- TMEM lane base+i).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// UMMA shared-memory matrix descriptor: K-major operand, 128-byte swizzle, rows of 64 bf16 (128 B),
// 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout SWIZZLE_128B=2 [61,64)).
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1) << 16;                 // LBO (unused for swizzled K-major; canonical value 1)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;         // SBO = 1024 B
    d |= static_cast<uint64_t>(1) << 46;                 // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;                 // SWIZZLE_128B
    return d;
}
// --------------------------------------------------------------------------------------------
// CTA pair (cta_group::2): two CTAs of one cluster (the two SMs of a TPC) run ONE 256-row MMA; each stages its own 128
// rows of A and HALF of the B tile, so the shared-memory traffic per SM per flop drops by a third at block_n = 256.
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {       // every thread of both CTAs
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
// arrive on an mbarrier of another CTA of the cluster (address from mapa_shared), release at cluster scope
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];\n" ::"r"(bar_cluster) : "memory");
}
// wait on a LOCAL mbarrier whose arrivals may come from the other CTA of the cluster (acquire at cluster scope); bounded
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    const long long t0 = clock64();
    while (true) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred P;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, P;\n\t}\n"
            : "=r"(ok)
            : "r"(a), "r"(parity)
            : "memory");
        if (ok) return;
        if (clock64() - t0 > 4000000000LL) {
            printf("tmae: cluster mbarrier wait timed out (block %d thread %d parity %u)\n", blockIdx.x, threadIdx.x, parity);
            __trap();
        }
    }
}
// TMA load into THIS CTA's shared memory whose completion bytes are signalled on an mbarrier of either CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(uint32_t smem_dst, const void* tmap, uint32_t bar_cluster, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
            "r"(smem_dst),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t smem_dst, const void* tmap, uint32_t bar_cluster, int32_t c0, int32_t c1,
                                                 int32_t c2, int32_t c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::
            "r"(smem_dst),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {   // one warp of EACH CTA of the pair
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "r"(ncols) : "memory");
}
// issued by ONE thread of the leader CTA (cluster rank 0): M = 256 across the pair
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the mbarrier at the same shared-memory offset in every CTA of `cta_mask` once the MMAs issued so far are done
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(bar),
                 "h"(cta_mask)
                 : "memory");
}

// Instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=bf16, both K-major, dense.
__host__ __device__ inline uint32_t umma_idesc_bf16_f32(int M, int N) {
    uint32_t d = 0;
    d |= 1u << 4;                        // c_format = F32
    d |= 1u << 7;                        // a_format = BF16
    d |= 1u << 10;                       // b_format = BF16
    d |= static_cast<uint32_t>(N >> 3) << 17;
    d |= static_cast<uint32_t>(M >> 4) << 24;
    return d;
}

}  // namespace tmae
