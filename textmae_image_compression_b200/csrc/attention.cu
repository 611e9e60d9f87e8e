// Fused softmax attention over the visible tokens of one image and one head (timm 0.4.5 Attention.forward as
// used by the encoder blocks, MCM.py:313-322, 629-630):  softmax((q k^T) * hd^-0.5) v, head_dim = 64.
// Three kernels:
//   attention_tc_kernel   (default, Tp <= 384) tcgen05 / TMEM / TMA: persistent, warp-specialised, see its header below.
//   attention_kernel      mma.sync m16n8k16 + ldmatrix, one CTA per (image, head), K and V of all keys in shared memory,
//                         online softmax in registers: the fallback for longer sequences and the A/B partner
//                         (TMAE_NO_TC_ATTN=1).
//   attention_f32_kernel  fp32 CUDA-core attention of the precise (conformance) modes.
#include <math.h>

#include <cuda.h>

#include "common.cuh"
#include "kernels.h"

namespace tmae {

namespace {

constexpr int HD = 64;
constexpr int KPITCH = HD + 8;        // bf16 elements per K row in smem: 36 words -> conflict-free B-fragment loads
constexpr int kAttnWarps = 5;          // T = 65 (K = 64 kept patches + cls) is 5 query tiles of 16: one per warp, one round
constexpr int kAttnThreads = 32 * kAttnWarps;
// head dim 32 (the MAE decoder blocks, T = L + 1 up to 1025): pitch 40 elements (20 words: the 8 rows of an ldmatrix tile
// still fall in distinct bank groups), 8 warps and <= 64 registers (4 CTAs per SM at T = 197; a CTA holds all keys and its
// warps' Q tiles, (2 * 1040 + 8 * 16) * 40 * 2 B = 172.5 KiB at T = 1025, so there one CTA fills an SM's shared memory)
constexpr int kAttn32Warps = 8;

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}

// qkv: bf16 [N*T, 3C] with columns [3][H][64] (timm reshape (B,T,3,H,hd)); out: bf16 [N*T, C] columns [H][64].
// K and V of all keys are staged ROW-major (pitch 72 elements: the 8 rows of an ldmatrix tile fall in distinct bank
// groups) together with each warp's 16-row Q tile, all in one round of independent 16-byte global loads; every MMA
// fragment then comes from ldmatrix (Q, K plain; V .trans): no transposed copy of V, no scalar shared-memory traffic
// and no Q registers held across the key loop (<= 64 registers -> 6 CTAs / 30 warps per SM, 888 slots >= the 768
// (image, head) CTAs of batch 64: one wave, one query tile per warp).
// Templated on the head dim D (64: the encoder, 32: the MAE decoder of the synthesis plan) and the warp count W; the D = 64,
// W = 5 instance is the encoder's kernel.
template <int D, int W, int MINB>
__global__ void __launch_bounds__(32 * W, MINB)
attention_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int T, int Tp, int H, int C,
                 float scale_log2e) {
    constexpr int HD = D, KPITCH = D + 8, kAttnWarps = W, kAttnThreads = 32 * W;
    pdl_wait();
    pdl_launch_dependents();
    extern __shared__ __align__(16) uint8_t smem_attn[];
    __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem_attn);            // [Tp][KPITCH]
    __nv_bfloat16* sV = sK + (size_t)Tp * KPITCH;                                // [Tp][KPITCH]
    __nv_bfloat16* sQ = sV + (size_t)Tp * KPITCH;                                // [kAttnWarps][16][KPITCH]
    const int n = blockIdx.x / H, h = blockIdx.x - n * H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const size_t ld = (size_t)3 * C;
    const __nv_bfloat16* base = qkv + (size_t)n * T * ld + (size_t)h * HD;
    __nv_bfloat16* myQ = sQ + (size_t)warp * 16 * KPITCH;

    // this warp's Q tile: 16 rows x HD dims = 2 HD 16-byte chunks, HD / 16 per lane (rows >= T are zero)
    auto stage_q = [&](int q0) {
#pragma unroll
        for (int i = 0; i < HD / 16; ++i) {
            const int e = i * 32 + lane, r = e / (HD / 8), c8 = (e % (HD / 8)) * 8;
            uint4 qv = make_uint4(0, 0, 0, 0);
            if (q0 + r < T) qv = *reinterpret_cast<const uint4*>(base + (size_t)(q0 + r) * ld + c8);
            *reinterpret_cast<uint4*>(myQ + r * KPITCH + c8) = qv;
        }
    };
    const int q_tiles = Tp / 16;
    if (warp < q_tiles) stage_q(warp * 16);
    // ---- stage K and V for all keys (16-byte chunks, coalesced: 8 threads per key row); zero the padding ----
#pragma unroll 4
    for (int e = tid; e < Tp * (HD / 8); e += kAttnThreads) {
        const int key = e / (HD / 8), c8 = (e - key * (HD / 8)) * 8;
        uint4 kv = make_uint4(0, 0, 0, 0), vv = make_uint4(0, 0, 0, 0);
        if (key < T) {
            kv = *reinterpret_cast<const uint4*>(base + (size_t)key * ld + C + c8);
            vv = *reinterpret_cast<const uint4*>(base + (size_t)key * ld + 2 * C + c8);
        }
        *reinterpret_cast<uint4*>(sK + (size_t)key * KPITCH + c8) = kv;
        *reinterpret_cast<uint4*>(sV + (size_t)key * KPITCH + c8) = vv;
    }
    __syncthreads();

    const uint32_t sK_a = smem_u32(sK), sV_a = smem_u32(sV), sQ_a = smem_u32(myQ);
    // per-lane ldmatrix row addresses (bytes) relative to the first key of a chunk
    //   K (plain):  matrix j = lane >> 3 covers d columns [8j, 8j+8) of keys (lane & 7)           (+32 columns for the 2nd load)
    //   V (.trans): matrices (keys 0-7, d0) (keys 8-15, d0) (keys 0-7, d0+8) (keys 8-15, d0+8)
    //   Q (plain):  matrices (rows 0-7, k0) (rows 8-15, k0) (rows 0-7, k0+8) (rows 8-15, k0+8) = a0..a3 of one k-step
    const uint32_t k_lane = (uint32_t)(((lane & 7) * KPITCH + (lane >> 3) * 8) * 2);
    const uint32_t v_lane = (uint32_t)((((lane & 7) + ((lane >> 3) & 1) * 8) * KPITCH + (lane >> 4) * 8) * 2);

    for (int qt = warp; qt < q_tiles; qt += kAttnWarps) {
        const int q0 = qt * 16;
        if (qt != warp) {                          // later rounds (T > 80): restage this warp's Q slot
            __syncwarp();
            stage_q(q0);
            __syncwarp();
        }
        float o[HD / 8][4];
#pragma unroll
        for (int i = 0; i < HD / 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
        float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;     // rows g and g+8

        for (int k0 = 0; k0 < Tp; k0 += 16) {
            // S chunk = Q (16x64) * K[k0..k0+16)^T : two n-tiles of 8 keys
            float sacc[2][4];
            sacc[0][0] = sacc[0][1] = sacc[0][2] = sacc[0][3] = 0.f;
            sacc[1][0] = sacc[1][1] = sacc[1][2] = sacc[1][3] = 0.f;
            const uint32_t ka = sK_a + (uint32_t)(k0 * KPITCH * 2) + k_lane;
#pragma unroll
            for (int hk = 0; hk < HD / 32; ++hk) {  // d 0..31 (k-steps 0, 1), then d 32..63 (k-steps 2, 3)
                uint32_t kb0[4], kb1[4], qa[4];
                ldmatrix_x4(kb0, ka + (uint32_t)(hk * 64));                               // keys k0 .. k0+7
                ldmatrix_x4(kb1, ka + (uint32_t)(8 * KPITCH * 2 + hk * 64));              // keys k0+8 .. k0+15
                ldmatrix_x4(qa, sQ_a + v_lane + (uint32_t)(hk * 64));                     // k-step 2 hk
                mma_bf16_16816(sacc[0], qa, kb0[0], kb0[1]);
                mma_bf16_16816(sacc[1], qa, kb1[0], kb1[1]);
                ldmatrix_x4(qa, sQ_a + v_lane + (uint32_t)(hk * 64 + 32));                // k-step 2 hk + 1
                mma_bf16_16816(sacc[0], qa, kb0[2], kb0[3]);
                mma_bf16_16816(sacc[1], qa, kb1[2], kb1[3]);
            }
            // scale (log2 domain), mask padded keys
            float cmax0 = -INFINITY, cmax1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const int key = k0 + nt * 8 + 2 * t;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const bool ok = (key + (i & 1)) < T;
                    sacc[nt][i] = ok ? sacc[nt][i] * scale_log2e : -INFINITY;
                }
                cmax0 = fmaxf(cmax0, fmaxf(sacc[nt][0], sacc[nt][1]));
                cmax1 = fmaxf(cmax1, fmaxf(sacc[nt][2], sacc[nt][3]));
            }
            cmax0 = fmaxf(cmax0, __shfl_xor_sync(0xffffffffu, cmax0, 1));
            cmax0 = fmaxf(cmax0, __shfl_xor_sync(0xffffffffu, cmax0, 2));
            cmax1 = fmaxf(cmax1, __shfl_xor_sync(0xffffffffu, cmax1, 1));
            cmax1 = fmaxf(cmax1, __shfl_xor_sync(0xffffffffu, cmax1, 2));
            const float nm0 = fmaxf(m0, cmax0), nm1 = fmaxf(m1, cmax1);   // finite: key 0 of chunk 0 is always valid
            const float corr0 = exp2f(m0 - nm0), corr1 = exp2f(m1 - nm1);
            m0 = nm0; m1 = nm1;
            float rs0 = 0.f, rs1 = 0.f;
            uint32_t pa[4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float p0 = exp2f(sacc[nt][0] - nm0), p1 = exp2f(sacc[nt][1] - nm0);
                const float p2 = exp2f(sacc[nt][2] - nm1), p3 = exp2f(sacc[nt][3] - nm1);
                rs0 += p0 + p1;
                rs1 += p2 + p3;
                pa[nt * 2 + 0] = pack_bf16x2(p0, p1);      // rows g   : a0 (keys 0-7) / a2 (keys 8-15)
                pa[nt * 2 + 1] = pack_bf16x2(p2, p3);      // rows g+8 : a1 / a3
            }
            l0 = l0 * corr0 + rs0;
            l1 = l1 * corr1 + rs1;
#pragma unroll
            for (int dt = 0; dt < HD / 8; ++dt) {
                o[dt][0] *= corr0; o[dt][1] *= corr0; o[dt][2] *= corr1; o[dt][3] *= corr1;
            }
            // O += P (16 x 16 keys) * V[k0..k0+16) (16 keys x HD): one transposing ldmatrix per pair of 8-wide d tiles
            const uint32_t va = sV_a + (uint32_t)(k0 * KPITCH * 2) + v_lane;
#pragma unroll
            for (int dp = 0; dp < HD / 16; ++dp) {
                uint32_t vb[4];
                ldmatrix_x4_trans(vb, va + (uint32_t)(dp * 32));
                mma_bf16_16816(o[2 * dp], pa, vb[0], vb[1]);
                mma_bf16_16816(o[2 * dp + 1], pa, vb[2], vb[3]);
            }
        }
        // row sums live per quad: reduce across the 4 lanes that share a row
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
        l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        const float inv0 = 1.f / l0, inv1 = 1.f / l1;
        const int r0 = q0 + g, r1 = q0 + g + 8;
        __nv_bfloat16* obase = out + (size_t)n * T * C + (size_t)h * HD;
#pragma unroll
        for (int dt = 0; dt < HD / 8; ++dt) {
            const int c = dt * 8 + 2 * t;
            if (r0 < T) *reinterpret_cast<uint32_t*>(obase + (size_t)r0 * C + c) = pack_bf16x2(o[dt][0] * inv0, o[dt][1] * inv0);
            if (r1 < T) *reinterpret_cast<uint32_t*>(obase + (size_t)r1 * C + c) = pack_bf16x2(o[dt][2] * inv1, o[dt][3] * inv1);
        }
    }
}

inline int attn_tp(int T) { return (T + 15) / 16 * 16; }
inline size_t attn_smem(int T, int hd = HD, int warps = kAttnWarps) {
    const int Tp = attn_tp(T);
    return ((size_t)2 * Tp + (size_t)warps * 16) * (hd + 8) * sizeof(__nv_bfloat16);
}
#define ATTN64 attention_kernel<64, kAttnWarps, 6>
#define ATTN32 attention_kernel<32, kAttn32Warps, 4>

// ---------------------------------------------------------------------------------------------------------
// Precise mode (TMAE_FLAG_PRECISE_ALL): fp32 softmax attention on CUDA cores.  q, k, v arrive as split-bf16 plane pairs
// (hi + lo = 16 mantissa bits) from the precise QKV GEMM; scores, softmax (expf, like the reference's fp32 softmax) and
// the PV sum run in fp32; the result leaves as a plane pair for the precise proj GEMM.  One CTA per (image, head):
// K (pitch 65, conflict-free for lane = key) and V (lane = dim) of all keys in shared memory, one warp per query row.
// This op is 0.8-3 % of the path's FLOPs; precise mode trades throughput for reference-exact symbols.
// ---------------------------------------------------------------------------------------------------------
constexpr int kAttnF32Warps = 8;
constexpr int KP32 = HD + 1;
__global__ void __launch_bounds__(32 * kAttnF32Warps)
attention_f32_kernel(const __nv_bfloat16* __restrict__ qkv, long long qkv_lo, __nv_bfloat16* __restrict__ out, long long out_lo,
                     int T, int H, int C, float scale) {
    pdl_wait();
    pdl_launch_dependents();
    extern __shared__ __align__(16) uint8_t smem_attn[];
    float* sK = reinterpret_cast<float*>(smem_attn);                 // [T][65]
    float* sV = sK + (size_t)T * KP32;                               // [T][64]
    float* sQ = sV + (size_t)T * HD;                                 // [warps][64]
    float* sP = sQ + kAttnF32Warps * HD;                             // [warps][T]
    const int n = blockIdx.x / H, h = blockIdx.x - n * H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t ld = (size_t)3 * C;
    const __nv_bfloat16* base = qkv + (size_t)n * T * ld + (size_t)h * HD;
    auto ldf = [&](const __nv_bfloat16* p) { return load_bf16_planes(p, qkv_lo); };
    for (int e = tid; e < T * HD; e += blockDim.x) {
        const int key = e / HD, d = e - key * HD;
        sK[key * KP32 + d] = ldf(base + (size_t)key * ld + C + d);
        sV[key * HD + d] = ldf(base + (size_t)key * ld + 2 * C + d);
    }
    __syncthreads();
    float* myQ = sQ + warp * HD;
    float* myP = sP + (size_t)warp * T;
    for (int q = warp; q < T; q += kAttnF32Warps) {
        myQ[lane] = ldf(base + (size_t)q * ld + lane);
        myQ[lane + 32] = ldf(base + (size_t)q * ld + lane + 32);
        __syncwarp();
        float mx = -INFINITY;
        for (int j = lane; j < T; j += 32) {
            const float* kr = sK + j * KP32;
            float acc = 0.f;
#pragma unroll 16
            for (int d = 0; d < HD; ++d) acc = fmaf(myQ[d], kr[d], acc);
            acc *= scale;
            myP[j] = acc;
            mx = fmaxf(mx, acc);
        }
        mx = warp_max(mx);
        float sum = 0.f;
        for (int j = lane; j < T; j += 32) {
            const float pj = expf(myP[j] - mx);
            myP[j] = pj;
            sum += pj;
        }
        sum = warp_sum(sum);
        __syncwarp();
        float o0 = 0.f, o1 = 0.f;
        for (int j = 0; j < T; ++j) {
            const float pj = myP[j];
            o0 = fmaf(pj, sV[j * HD + lane], o0);
            o1 = fmaf(pj, sV[j * HD + lane + 32], o1);
        }
        const float inv = 1.f / sum;
        o0 *= inv; o1 *= inv;
        __nv_bfloat16* dst = out + ((size_t)n * T + q) * C + (size_t)h * HD;
        store_bf16_planes(dst + lane, out_lo, o0);
        store_bf16_planes(dst + lane + 32, out_lo, o1);
        __syncwarp();
    }
}
inline size_t attn_f32_smem(int T) {
    return ((size_t)T * KP32 + (size_t)T * HD + (size_t)kAttnF32Warps * HD + (size_t)kAttnF32Warps * T) * sizeof(float);
}

// ---------------------------------------------------------------------------------------------------------
// tcgen05 attention (bf16 mode, Tp <= 384): a PERSISTENT, warp-specialised kernel - one CTA per SM walks a list of
// (image, head, query tile) items; the pieces of consecutive items overlap:
//   warp 0    TMA producer: Q [<=128 x 64], K [Tp x 64], V [Tp x 64] boxes of the qkv matrix into an nst-stage ring
//             (all three SWIZZLE_128B; V is consumed as the MN-major B operand exactly as TMA wrote it - no transpose)
//   warp 1    MMA issuer: S = Q K^T (M 128, N Tp, K 64) into TMEM buffer b, O = P V (M 128, N 64, K Tp) into O buffer b;
//             S of item i+1 is issued BEFORE waiting for the softmax of item i (two S / O / P buffers when Tp <= 192)
//   warps 2-5 / 6-9   two softmax groups (128 threads = 128 TMEM lanes = 128 query rows) taking alternate items: read the S
//             row with tcgen05.ld, max / exp2 / sum in registers (no shuffles), write P as the K-major 128B-swizzled A operand
//             of the second MMA, then read O, scale by 1 / sum and store the bf16 row.
// Barriers per item: full/empty (stage), s_ready, p_ready (128 arrivals), o_ready, o_free (128 arrivals).  WAR hazards on
// S (next S MMA vs. this softmax's loads) and P (next softmax's stores vs. this PV MMA) are covered by program order of
// the issuing warp / the owning group, see the loop comments.
// Rows >= T of a tile belong to the next image (or are zero-filled at the end of the tensor): as keys they are masked in the
// softmax, as queries they are computed on whatever the tile holds and never stored.
// ---------------------------------------------------------------------------------------------------------
constexpr int kAttnTcThreads = 320;
constexpr int kAttnTcMaxTp = 384;
constexpr int kAttnTcMaxStages = 3;

struct AttnTcParams {
    int T, Tp, H, C;
    int n_items, q_tiles;
    int duo;                  // 1: two heads per 128-row tile (T - 1 = 64 patch queries each), S = [128 x 2 Tp]; cls queries on the tail warp
    int Tpt;                  // key columns of the S tile: Tp, or 2 Tp in duo mode
    int tail_rows;            // query rows past the last full 128-row tile (T = 257: the 257th) computed by the tail warp on CUDA cores
    int nbuf;                 // 2: double-buffered S / O / P and both softmax groups; 1: single (Tp > 192)
    int nst;                  // Q/K/V stages
    int qrows, krows, kloads; // TMA boxes: Q rows, K/V rows per load, loads per K/V tile
    int atoms;                // 64-key atoms of the P tile
    uint32_t qreg, kreg;      // bytes reserved per Q / K / V tile (multiples of 1024)
    uint32_t s_stride, o_col0, tmem_cols;
    float scale_log2e;
    long long* dbg;           // bring-up: [item][16] clock64 stamps of CTA 0 (TMAE_ATTN_TIMING=1), else nullptr
};

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// MN-major (transposed) B operand, 128-byte swizzle: rows of the K dimension are 128 B apart, 8-row groups 1024 B apart
// (cute::UMMA canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units; one 64-element MN block, so LBO is unused).
__device__ __forceinline__ uint64_t umma_smem_desc_mn_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

// WGS = softmax groups per CTA.  2: one 320-thread CTA per SM with double-buffered S / O / P (or 1 buffer for long rows).
// 1 ("lite", Tp <= 96): 192 threads, one buffer, two pipeline stages, 256 TMEM columns, <= 93 KB shared memory - two such CTAs
// share an SM, or one of them shares it with a GEMM CTA of another stream (multi-stream mode, TMAE_FLAG_SHARE_SM).
// DUO = the two-heads-per-tile experiment (compile-time, so the plain forms carry none of its address arithmetic).
template <int NCH, int WGS, bool DUO = false>      // S row held in NCH x 32 registers (Tp <= 32 NCH); 0 = streamed from tensor memory in two passes
__global__ void __launch_bounds__(64 + 128 * WGS + (WGS == 2 ? 32 : 0), WGS == 1 ? 2 : 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_kv,
                    const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, const AttnTcParams p) {
    constexpr bool kTailWarp = WGS == 2;          // one more warp: the few query rows past the last full tile, on CUDA cores
    pdl_launch_dependents();
    extern __shared__ __align__(1024) uint8_t smem_tc[];
    const uint32_t stage_bytes = p.qreg + 2u * p.kreg;
    const uint32_t smem0 = smem_u32(smem_tc);
    const uint32_t p_base = smem0 + (uint32_t)p.nst * stage_bytes;
    const uint32_t p_bytes = (uint32_t)p.atoms * 16384u;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_tc + (size_t)p.nst * stage_bytes + (size_t)p.nbuf * p_bytes);
    // full[3] empty[3] s_ready[2] p_ready[2] o_ready[2] o_free[2]
    const uint32_t bar0 = smem_u32(bars);
    auto bar_full = [&](int s) { return bar0 + 8u * (uint32_t)s; };
    auto bar_empty = [&](int s) { return bar0 + 8u * (uint32_t)(3 + s); };
    auto bar_sready = [&](int b) { return bar0 + 8u * (uint32_t)(6 + b); };
    auto bar_pready = [&](int b) { return bar0 + 8u * (uint32_t)(8 + b); };
    auto bar_oready = [&](int b) { return bar0 + 8u * (uint32_t)(10 + b); };
    auto bar_ofree = [&](int b) { return bar0 + 8u * (uint32_t)(12 + b); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);
    float* tail_p = reinterpret_cast<float*>(bars + 16);       // [<= 384] scores / probabilities of the tail warp's query row
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < 3; ++s) { mbar_init(&bars[s], 1); mbar_init(&bars[3 + s], kTailWarp ? 2 : 1); }   // empty: MMA commit (+ tail warp)
        for (int b = 0; b < 2; ++b) { mbar_init(&bars[6 + b], 1); mbar_init(&bars[8 + b], 128); mbar_init(&bars[10 + b], 1); mbar_init(&bars[12 + b], 128); }
        fence_barrier_init();
        tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_kv);
    }
    if (warp == 0) { tmem_alloc(tmem_slot, p.tmem_cols); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    pdl_wait();

    const int n_my = (p.n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const uint32_t kbytes = (uint32_t)p.Tp * 128u;

    if (warp == 0) {
        if (lane == 0) {
            for (int k = 0; k < n_my; ++k) {
                const int item = (int)blockIdx.x + k * (int)gridDim.x;
                const int qt = item % p.q_tiles, nh = item / p.q_tiles;
                const int hgroups = DUO ? p.H >> 1 : p.H;
                const int h = (nh % hgroups) << (DUO ? 1 : 0), n = nh / hgroups;
                const int st = k % p.nst;
                mbar_wait_a(bar_empty(st), (((uint32_t)(k / p.nst)) & 1u) ^ 1u);
                const uint32_t base = smem0 + (uint32_t)st * stage_bytes;
                const int row0 = n * p.T;
                if (DUO) {
                    // two heads: patch queries 1..T-1 of head h in tile rows 0..63, of head h+1 in rows 64..127; the keys / values
                    // of the two heads one after the other (Tp rows each)
                    mbar_arrive_expect_tx_a(bar_full(st), 2u * (uint32_t)p.qrows * 128u + 4u * kbytes);
                    for (int sidx = 0; sidx < 2; ++sidx) {
                        tma_load_2d_a(base + (uint32_t)sidx * 8192u, &map_q, bar_full(st), (h + sidx) * HD, row0 + 1);
                        tma_load_2d_a(base + p.qreg + (uint32_t)sidx * kbytes, &map_kv, bar_full(st), p.C + (h + sidx) * HD, row0);
                        tma_load_2d_a(base + p.qreg + p.kreg + (uint32_t)sidx * kbytes, &map_kv, bar_full(st), 2 * p.C + (h + sidx) * HD, row0);
                    }
                    continue;
                }
                mbar_arrive_expect_tx_a(bar_full(st), (uint32_t)p.qrows * 128u + 2u * kbytes);
                tma_load_2d_a(base, &map_q, bar_full(st), h * HD, row0 + qt * 128);
                for (int l = 0; l < p.kloads; ++l) {
                    tma_load_2d_a(base + p.qreg + (uint32_t)(l * p.krows) * 128u, &map_kv, bar_full(st), p.C + h * HD, row0 + l * p.krows);
                    tma_load_2d_a(base + p.qreg + p.kreg + (uint32_t)(l * p.krows) * 128u, &map_kv, bar_full(st), 2 * p.C + h * HD,
                                  row0 + l * p.krows);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc_pv = umma_idesc_bf16_f32(128, HD) | (1u << 16);            // B (= V) is MN-major
            auto issue_s = [&](int k) {
                const int st = k % p.nst, b = k % p.nbuf;
                mbar_wait_a(bar_full(st), ((uint32_t)(k / p.nst)) & 1u);
                tc_fence_after();
                if (p.dbg && blockIdx.x == 0) p.dbg[k * 16 + 0] = clock64();
                const uint32_t base = smem0 + (uint32_t)st * stage_bytes;
                const uint64_t dq = umma_smem_desc_sw128(base);
                for (int n0 = 0; n0 < p.Tpt; n0 += 256) {
                    const int nn = min(256, p.Tpt - n0);
                    const uint32_t idesc = umma_idesc_bf16_f32(128, nn);
                    const uint64_t dk = umma_smem_desc_sw128(base + p.qreg + (uint32_t)n0 * 128u);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_bf16(tmem + (uint32_t)b * p.s_stride + (uint32_t)n0, dq + (uint64_t)(2 * kk), dk + (uint64_t)(2 * kk), idesc, kk != 0 ? 1u : 0u);
                }
                umma_commit_a(bar_sready(b));
                if (p.dbg && blockIdx.x == 0) p.dbg[k * 16 + 1] = clock64();
            };
            if (n_my > 0 && p.nbuf == 2) issue_s(0);
            for (int k = 0; k < n_my; ++k) {
                const int st = k % p.nst, b = k % p.nbuf;
                const uint32_t use = (uint32_t)(k / p.nbuf);
                // S buffer of the item issued here was last read by the softmax of item k-1 (dual) / k-1 (single): its
                // p_ready was waited for below in the previous iteration, so the loads of that S row are complete.
                if (p.nbuf == 2) { if (k + 1 < n_my) issue_s(k + 1); }
                else issue_s(k);
                mbar_wait_a(bar_pready(b), use & 1u);                 // P of item k is in shared memory
                if (p.dbg && blockIdx.x == 0) p.dbg[k * 16 + 2] = clock64();
                mbar_wait_a(bar_ofree(b), (use & 1u) ^ 1u);           // O buffer b drained by the epilogue of item k - nbuf
                tc_fence_after();
                const uint32_t base = smem0 + (uint32_t)st * stage_bytes;
                const uint64_t dp = umma_smem_desc_sw128(p_base + (uint32_t)b * p_bytes);
                const uint64_t dv = umma_smem_desc_mn_sw128(base + p.qreg + p.kreg);
                const int ksteps = p.Tpt >> 4;
                for (int ks = 0; ks < ksteps; ++ks) {
                    const uint64_t a_desc = dp + (uint64_t)((uint32_t)(ks >> 2) * (16384u >> 4)) + (uint64_t)(2 * (ks & 3));
                    const uint64_t b_desc = dv + (uint64_t)((uint32_t)ks * (2048u >> 4));
                    umma_bf16(tmem + p.o_col0 + (uint32_t)b * 64u, a_desc, b_desc, idesc_pv, ks != 0 ? 1u : 0u);
                }
                umma_commit_a(bar_oready(b));
                umma_commit_a(bar_empty(st));                         // Q / K / V of this stage are no longer read
                if (p.dbg && blockIdx.x == 0) p.dbg[k * 16 + 3] = clock64();
            }
        }
    } else if (kTailWarp && warp == 2 + 4 * WGS) {
        // ===== tail warp: T = 128 q + r with r <= 8 (ViT-L: 257 = 2 x 128 + 1).  A third query tile for r rows would repeat
        // the whole K / V load and both MMAs; instead the item of the LAST full tile also computes those r rows here, on CUDA
        // cores, from the K / V tiles already in shared memory (swizzled as TMA wrote them): lanes = keys for q k^T, lanes =
        // dim pairs for p v.  Every item is waited for and released (empty has two arrivals), so the warp cannot run ahead.
        for (int k = 0; k < n_my; ++k) {
            const int item = (int)blockIdx.x + k * (int)gridDim.x;
            const int qt = item % p.q_tiles, nh = item / p.q_tiles;
            const int hgroups = DUO ? p.H >> 1 : p.H;
            const int h0 = (nh % hgroups) << (DUO ? 1 : 0), n = nh / hgroups;
            const int st = k % p.nst;
            mbar_wait_a(bar_full(st), ((uint32_t)(k / p.nst)) & 1u);
            if (p.tail_rows > 0 && qt == p.q_tiles - 1) {
                for (int tr = 0; tr < p.tail_rows; ++tr) {
                    // duo: tail row tr = the cls query (token 0) of head h0 + tr, against that head's keys; else token 128 q + tr
                    const int h = DUO ? h0 + tr : h0;
                    const int t = DUO ? 0 : p.q_tiles * 128 + tr;
                    const uint32_t kb = smem0 + (uint32_t)st * stage_bytes + p.qreg + (DUO ? (uint32_t)tr * kbytes : 0u), vb = kb + p.kreg;
                    const uint4* qg = reinterpret_cast<const uint4*>(qkv + (size_t)(n * p.T + t) * 3 * p.C + (size_t)h * HD);
                    float q[HD];
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint4 v = __ldg(qg + c);
                        const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            q[c * 8 + 2 * e] = __uint_as_float(w4[e] << 16);
                            q[c * 8 + 2 * e + 1] = __uint_as_float(w4[e] & 0xffff0000u);
                        }
                    }
                    // rolled loops (the scores live in shared memory, not in a register array): this warp's code must stay
                    // small - a fully unrolled version thrashed the instruction cache and cost more than the tile it saved
                    float mx = -INFINITY;
                    for (int j = lane; j < p.T; j += 32) {
                        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;        // four independent chains: the dot product is latency-bound
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            const float4 kv = lds128(kb + (uint32_t)j * 128u + ((((uint32_t)c) ^ ((uint32_t)j & 7u)) << 4));
                            const uint32_t w4[4] = {__float_as_uint(kv.x), __float_as_uint(kv.y), __float_as_uint(kv.z), __float_as_uint(kv.w)};
                            a0 = fmaf(q[c * 8 + 0], __uint_as_float(w4[0] << 16), a0);
                            a1 = fmaf(q[c * 8 + 1], __uint_as_float(w4[0] & 0xffff0000u), a1);
                            a2 = fmaf(q[c * 8 + 2], __uint_as_float(w4[1] << 16), a2);
                            a3 = fmaf(q[c * 8 + 3], __uint_as_float(w4[1] & 0xffff0000u), a3);
                            a0 = fmaf(q[c * 8 + 4], __uint_as_float(w4[2] << 16), a0);
                            a1 = fmaf(q[c * 8 + 5], __uint_as_float(w4[2] & 0xffff0000u), a1);
                            a2 = fmaf(q[c * 8 + 6], __uint_as_float(w4[3] << 16), a2);
                            a3 = fmaf(q[c * 8 + 7], __uint_as_float(w4[3] & 0xffff0000u), a3);
                        }
                        const float sv = ((a0 + a1) + (a2 + a3)) * p.scale_log2e;
                        tail_p[j] = sv;
                        mx = fmaxf(mx, sv);
                    }
                    mx = warp_max(mx);
                    float sum = 0.f;
                    const int t8 = (p.T + 7) & ~7;
                    for (int j = lane; j < t8; j += 32) {
                        // P is rounded to bf16 before the second product, like the tensor-core path does
                        const float pe = j < p.T ? ex2_approx(tail_p[j] - mx) : 0.f;
                        sum += pe;
                        tail_p[j] = __bfloat162float(__float2bfloat16(pe));
                    }
                    sum = warp_sum(sum);
                    __syncwarp();
                    // p v: lanes = dim pairs, eight keys per step (rows up to the next multiple of 8 exist in the tile, their p is 0)
                    float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;
                    const uint32_t vlane = (((uint32_t)lane & 3u) * 4u);
                    for (int j0 = 0; j0 < t8; j0 += 8) {
                        uint32_t vw[8];
                        float pj[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const uint32_t jj = (uint32_t)(j0 + u);
                            asm volatile("ld.shared.b32 %0, [%1];\n" : "=r"(vw[u])
                                         : "r"(vb + jj * 128u + ((((uint32_t)lane >> 2) ^ (jj & 7u)) << 4) + vlane));
                            pj[u] = tail_p[j0 + u];
                        }
#pragma unroll
                        for (int u = 0; u < 8; u += 2) {
                            o0 = fmaf(pj[u], __uint_as_float(vw[u] << 16), o0);
                            o1 = fmaf(pj[u], __uint_as_float(vw[u] & 0xffff0000u), o1);
                            o2 = fmaf(pj[u + 1], __uint_as_float(vw[u + 1] << 16), o2);
                            o3 = fmaf(pj[u + 1], __uint_as_float(vw[u + 1] & 0xffff0000u), o3);
                        }
                    }
                    o0 += o2; o1 += o3;
                    __syncwarp();                                     // tail_p is rewritten by the next tail row
                    const float inv = 1.f / sum;
                    *reinterpret_cast<uint32_t*>(out + (size_t)(n * p.T + t) * p.C + (size_t)h * HD + 2 * lane) = pack_bf16x2(o0 * inv, o1 * inv);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars[3 + st]);
        }
    } else {
        const int g = (warp - 2) >> 2;                                // softmax group
        const int quad = warp & 3;                                    // TMEM lane quadrant this warp may access
        const int row = quad * 32 + lane;
        const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
        if (g < p.nbuf) {
            for (int k = g; k < n_my; k += p.nbuf) {
                const int item = (int)blockIdx.x + k * (int)gridDim.x;
                const int qt = item % p.q_tiles, nh = item / p.q_tiles;
                const int hgroups = DUO ? p.H >> 1 : p.H;
                const int sub = DUO ? quad >> 1 : 0;                  // duo: tile rows 0..63 = head h, 64..127 = head h + 1
                const int h = ((nh % hgroups) << (DUO ? 1 : 0)) + sub, n = nh / hgroups;
                const int b = k % p.nbuf;
                const uint32_t use = (uint32_t)(k / p.nbuf);
                const int q0 = DUO ? 1 - sub * 64 : qt * 128;         // token of tile row r = q0 + r
                const bool valid = q0 + row < p.T;
                const int lo = DUO ? sub * p.Tp : 0, hi = lo + p.T;               // this row's keys are S columns [lo, hi) (warp-uniform)
                const uint32_t s_addr = tmem + lane_off + (uint32_t)b * p.s_stride;
                const bool stamp = p.dbg && blockIdx.x == 0 && row == 0;
                if (stamp) p.dbg[k * 16 + 4] = clock64();
                mbar_wait_a(bar_sready(b), use & 1u);
                tc_fence_after();
                if (stamp) p.dbg[k * 16 + 5] = clock64();
                const uint32_t prow = p_base + (uint32_t)b * p_bytes + (uint32_t)row * 128u;
                const uint32_t rsw = (uint32_t)(row & 7);
                float mx = -INFINITY, sum = 0.f;
                // 32 S values at key columns [c0, c0 + 32): running maximum / exp2, row sum, bf16 P into the swizzled A tile.
                // Columns are masked only in the 8-column group that straddles T; groups past T are written as zeros.
                auto chunk_max = [&](const uint32_t (&sv)[32], int c0) {
                    if (c0 >= lo && c0 + 32 <= hi) {
                        float m0 = __uint_as_float(sv[0]), m1 = __uint_as_float(sv[1]), m2 = __uint_as_float(sv[2]), m3 = __uint_as_float(sv[3]);
#pragma unroll
                        for (int i = 4; i < 32; i += 4) {
                            m0 = fmaxf(m0, __uint_as_float(sv[i])); m1 = fmaxf(m1, __uint_as_float(sv[i + 1]));
                            m2 = fmaxf(m2, __uint_as_float(sv[i + 2])); m3 = fmaxf(m3, __uint_as_float(sv[i + 3]));
                        }
                        mx = fmaxf(mx, fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)));
                    } else {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int cq = c0 + q * 8;
                            if (cq + 8 > lo && cq < hi) {
#pragma unroll
                                for (int i = 0; i < 8; ++i) if (cq + i >= lo && cq + i < hi) mx = fmaxf(mx, __uint_as_float(sv[q * 8 + i]));
                            }
                        }
                    }
                };
                auto chunk_exp = [&](const uint32_t (&sv)[32], int c0, float mxs) {
                    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        uint32_t pk[4] = {0u, 0u, 0u, 0u};
                        const int cq = c0 + q * 8;
                        if (cq >= lo && cq + 8 <= hi) {
                            float e[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) e[i] = ex2_approx(fmaf(__uint_as_float(sv[q * 8 + i]), p.scale_log2e, -mxs));
                            s0 += e[0] + e[4]; s1 += e[1] + e[5]; s2 += e[2] + e[6]; s3 += e[3] + e[7];
#pragma unroll
                            for (int i = 0; i < 4; ++i) pk[i] = pack_bf16x2(e[2 * i], e[2 * i + 1]);
                        } else if (cq + 8 > lo && cq < hi) {
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int c = cq + 2 * i;
                                const float p0 = (c >= lo && c < hi) ? ex2_approx(fmaf(__uint_as_float(sv[q * 8 + 2 * i]), p.scale_log2e, -mxs)) : 0.f;
                                const float p1 = (c + 1 >= lo && c + 1 < hi) ? ex2_approx(fmaf(__uint_as_float(sv[q * 8 + 2 * i + 1]), p.scale_log2e, -mxs)) : 0.f;
                                s0 += p0 + p1;
                                pk[i] = pack_bf16x2(p0, p1);
                            }
                        }
                        if (cq < p.Tpt) {
                            if constexpr (DUO)     // c0 is not 32-aligned: 64-key atom cq / 64, 16-byte chunk (cq % 64) / 8 per group
                                sts128(prow + (uint32_t)(cq >> 6) * 16384u + (((((uint32_t)cq & 63u) >> 3) ^ rsw) << 4), pk[0], pk[1], pk[2], pk[3]);
                            else                   // c0 % 32 == 0: the four groups of a chunk stay inside one atom
                                sts128(prow + (uint32_t)(c0 >> 6) * 16384u + ((((((uint32_t)c0 & 63u) >> 3) + (uint32_t)q) ^ rsw) << 4), pk[0], pk[1],
                                       pk[2], pk[3]);
                        }
                    }
                    sum += (s0 + s1) + (s2 + s3);
                };
                if constexpr (NCH > 0) {
                    // the whole S row in registers: one round of TMEM loads, one wait
                    uint32_t sv[NCH][32];
#pragma unroll
                    for (int c = 0; c < NCH; ++c) tmem_ld_32x32b_x32(s_addr + (uint32_t)(lo + 32 * c), sv[c]);   // this row's own keys
                    tmem_ld_wait();
                    if (stamp) p.dbg[k * 16 + 6] = clock64();
                    if (valid) {
#pragma unroll
                        for (int c = 0; c < NCH; ++c) if (32 * c < p.Tp) chunk_max(sv[c], lo + 32 * c);
                        const float mxs = mx * p.scale_log2e;
#pragma unroll
                        for (int c = 0; c < NCH; ++c) if (32 * c < p.Tp) chunk_exp(sv[c], lo + 32 * c, mxs);
                        if constexpr (DUO) {                          // block-diagonal P: zeros against the other head's keys
                            const int olo = p.Tp - lo;
                            for (int cq = olo; cq < olo + p.Tp; cq += 8)
                                sts128(prow + (uint32_t)(cq >> 6) * 16384u + (((((uint32_t)cq & 63u) >> 3) ^ rsw) << 4), 0u, 0u, 0u, 0u);
                        }
                    }
                } else {
                    // long rows: two passes over tensor memory, the load of the next 32 columns in flight while this one is used
                    uint32_t sa[32], sb[32];
                    float mxs = 0.f;
                    for (int pass = 0; pass < 2; ++pass) {
                        tmem_ld_32x32b_x32(s_addr, sa);
                        tmem_ld_wait();
                        for (int c0 = 0; c0 < p.Tpt; c0 += 64) {
                            const bool has_b = c0 + 32 < p.Tpt, has_a2 = c0 + 64 < p.Tpt;
                            if (has_b) tmem_ld_32x32b_x32(s_addr + (uint32_t)(c0 + 32), sb);
                            if (valid) { if (pass == 0) chunk_max(sa, c0); else chunk_exp(sa, c0, mxs); }
                            tmem_ld_wait();
                            if (has_b) {
                                if (has_a2) tmem_ld_32x32b_x32(s_addr + (uint32_t)(c0 + 64), sa);
                                if (valid) { if (pass == 0) chunk_max(sb, c0 + 32); else chunk_exp(sb, c0 + 32, mxs); }
                                tmem_ld_wait();
                            }
                        }
                        mxs = mx * p.scale_log2e;
                    }
                }
                if (stamp) p.dbg[k * 16 + 7] = clock64();
                fence_proxy_async_smem();                             // P written through the generic proxy -> visible to the MMA
                tc_fence_before();                                    // this thread's S loads are ordered before the next S MMA
                mbar_arrive(&bars[8 + b]);
                if (stamp) p.dbg[k * 16 + 8] = clock64();
                // ---- epilogue: O row / sum -> bf16 ----
                mbar_wait_a(bar_oready(b), use & 1u);
                tc_fence_after();
                if (stamp) p.dbg[k * 16 + 9] = clock64();
                uint32_t o0[32], o1[32];
                tmem_ld_32x32b_x32(tmem + lane_off + p.o_col0 + (uint32_t)b * 64u, o0);
                tmem_ld_32x32b_x32(tmem + lane_off + p.o_col0 + (uint32_t)b * 64u + 32u, o1);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(&bars[12 + b]);                           // O buffer b may be overwritten
                if (stamp) p.dbg[k * 16 + 10] = clock64();
                // O row * (1 / sum) -> bf16 into this group's (now idle) P tile, 128B-swizzled, then each warp copies its 32 rows
                // out with full 128-byte lines: lane -> (row l / 8 + 4 i, 16-byte chunk l % 8).
                const uint32_t stg = p_base + (uint32_t)b * p_bytes;
                if (valid) {
                    const float inv = 1.f / sum;
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        sts128(stg + (uint32_t)row * 128u + ((((uint32_t)c) ^ rsw) << 4),
                               pack_bf16x2(__uint_as_float(o0[8 * c]) * inv, __uint_as_float(o0[8 * c + 1]) * inv),
                               pack_bf16x2(__uint_as_float(o0[8 * c + 2]) * inv, __uint_as_float(o0[8 * c + 3]) * inv),
                               pack_bf16x2(__uint_as_float(o0[8 * c + 4]) * inv, __uint_as_float(o0[8 * c + 5]) * inv),
                               pack_bf16x2(__uint_as_float(o0[8 * c + 6]) * inv, __uint_as_float(o0[8 * c + 7]) * inv));
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        sts128(stg + (uint32_t)row * 128u + ((((uint32_t)(c + 4)) ^ rsw) << 4),
                               pack_bf16x2(__uint_as_float(o1[8 * c]) * inv, __uint_as_float(o1[8 * c + 1]) * inv),
                               pack_bf16x2(__uint_as_float(o1[8 * c + 2]) * inv, __uint_as_float(o1[8 * c + 3]) * inv),
                               pack_bf16x2(__uint_as_float(o1[8 * c + 4]) * inv, __uint_as_float(o1[8 * c + 5]) * inv),
                               pack_bf16x2(__uint_as_float(o1[8 * c + 6]) * inv, __uint_as_float(o1[8 * c + 7]) * inv));
                }
                __syncwarp();
                {
                    const int rows_left = p.T - q0 - quad * 32;                    // valid rows of this warp's 32
                    __nv_bfloat16* wdst = out + ((size_t)(n * p.T) + (size_t)(q0 + quad * 32)) * p.C + (size_t)h * HD;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int r = 4 * i + (lane >> 3);
                        if (r < rows_left) {
                            const uint32_t rr = (uint32_t)(quad * 32 + r);
                            const float4 v = lds128(stg + rr * 128u + ((((uint32_t)lane & 7u) ^ (rr & 7u)) << 4));
                            *reinterpret_cast<float4*>(wdst + (size_t)r * p.C + (lane & 7) * 8) = v;
                        }
                    }
                }
                __syncwarp();                                         // the tile is rewritten by this group's next softmax
                if (stamp) p.dbg[k * 16 + 11] = clock64();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 0) tmem_dealloc(tmem, p.tmem_cols);
}

// shared-memory / tensor-memory plan of the tcgen05 kernel for T tokens; returns false when it does not fit
inline bool attn_tc_plan(int T, int H, int C, int N, float scale, AttnTcParams* out, size_t* smem, bool lite = false, bool duo = false) {
    AttnTcParams p = {};
    const int Tp = attn_tp(T);
    if (Tp > kAttnTcMaxTp) return false;
    p.T = T; p.Tp = Tp; p.H = H; p.C = C;
    if (duo) {
        // two heads per tile: T - 1 = 64 patch queries per head (the K = 64 configuration), cls queries on the tail warp
        if (T != 65 || (H & 1) != 0 || lite) return false;
        p.duo = 1; p.Tpt = 2 * Tp;
        p.q_tiles = 1; p.tail_rows = 2;
        p.n_items = N * (H / 2);
        p.qrows = 64; p.kloads = 1; p.krows = Tp;
        p.atoms = (p.Tpt + 63) / 64;
        p.qreg = 16384;
        p.kreg = ((uint32_t)p.Tpt * 128u + 1023u) & ~1023u;
        const uint32_t sp2 = ((uint32_t)p.Tpt + 31u) & ~31u;
        const size_t stage2 = p.qreg + 2 * (size_t)p.kreg, pb2 = (size_t)p.atoms * 16384;
        p.nbuf = 2; p.nst = 2;
        if (2 * sp2 + 128 > 512 || 2 * stage2 + 2 * pb2 > 227 * 1024 - 2048) return false;
        p.s_stride = sp2; p.o_col0 = 2 * sp2; p.tmem_cols = 512;
        p.scale_log2e = scale * 1.4426950408889634f;
        *out = p;
        *smem = 2 * stage2 + 2 * pb2 + 2048;
        return true;
    }
    p.Tpt = Tp;
    p.q_tiles = (T + 127) / 128;
    p.tail_rows = 0;
    static const bool no_tail = getenv("TMAE_NO_ATTN_TAIL") != nullptr;
    if (!lite && !no_tail && T / 128 >= 1 && T % 128 != 0 && T % 128 <= 8) { p.q_tiles = T / 128; p.tail_rows = T % 128; }
    p.n_items = N * H * p.q_tiles;
    p.qrows = Tp < 128 ? Tp : 128;
    p.kloads = Tp <= 256 ? 1 : 2;
    p.krows = Tp / p.kloads;
    p.atoms = (Tp + 63) / 64;
    p.qreg = ((uint32_t)p.qrows * 128u + 1023u) & ~1023u;
    p.kreg = ((uint32_t)Tp * 128u + 1023u) & ~1023u;
    const uint32_t sp = ((uint32_t)Tp + 31u) & ~31u;
    const size_t limit = 227 * 1024 - 2048;                   // barriers, TMEM slot, tail-row scratch
    const size_t stage = p.qreg + 2 * (size_t)p.kreg, pb = (size_t)p.atoms * 16384;
    p.nbuf = (2 * sp + 128 <= 512 && 2 * stage + 2 * pb <= limit) ? 2 : 1;
    if (lite) p.nbuf = 1;
    if (stage + (size_t)p.nbuf * pb > limit) return false;
    int nst = (int)((limit - (size_t)p.nbuf * pb) / stage);
    p.nst = nst > kAttnTcMaxStages ? kAttnTcMaxStages : nst;
    if (lite && p.nst > 2) p.nst = 2;
    p.s_stride = sp;
    p.o_col0 = (uint32_t)p.nbuf * sp;
    const uint32_t need = p.o_col0 + (uint32_t)p.nbuf * 64u;
    p.tmem_cols = need <= 128 ? 128 : need <= 256 ? 256 : 512;
    if (need > 512) return false;
    p.scale_log2e = scale * 1.4426950408889634f;
    *out = p;
    *smem = (size_t)p.nst * stage + (size_t)p.nbuf * pb + 2048;
    return true;
}

}  // namespace

// The dynamic shared-memory limit is a property of the (process-global) kernel, not of a handle: it is raised to the
// device maximum once, so handles with different token counts can coexist in one process in any creation order.
cudaError_t attention_configure(int T) {
    if (attn_smem(T) > 227 * 1024) return cudaErrorInvalidValue;
    static cudaError_t once = [] {
        cudaError_t e = cudaFuncSetAttribute(ATTN64, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(attention_tc_kernel<3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(attention_tc_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(attention_tc_kernel<4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(attention_tc_kernel<0, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        return cudaFuncSetAttribute(attention_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    }();
    return once;
}

cudaError_t launch_attention(const __nv_bfloat16* qkv, __nv_bfloat16* out, int N, int T, int H, int C, float scale,
                             cudaStream_t st) {
    if (C != H * HD) return cudaErrorInvalidValue;
    const int Tp = attn_tp(T);
    TMAE_CARVEOUT_ONCE(ATTN64);
    return launch_k(ATTN64, dim3(N * H), dim3(kAttnThreads), attn_smem(T), st, true, qkv, out, T, Tp, H, C,
                    scale * 1.4426950408889634f);
}

bool attention_hd32_supported(int T) { return T >= 1 && attn_smem(T, 32, kAttn32Warps) <= 227 * 1024; }

cudaError_t launch_attention_hd32(const __nv_bfloat16* qkv, __nv_bfloat16* out, int N, int T, int H, float scale, cudaStream_t st) {
    if (!attention_hd32_supported(T)) return cudaErrorInvalidValue;
    static const cudaError_t configured = cudaFuncSetAttribute(ATTN32, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (configured != cudaSuccess) return configured;
    const int Tp = attn_tp(T);
    TMAE_CARVEOUT_ONCE(ATTN32);
    return launch_k(ATTN32, dim3(N * H), dim3(32 * kAttn32Warps), attn_smem(T, 32, kAttn32Warps), st, true, qkv, out, T, Tp, H, H * 32,
                    scale * 1.4426950408889634f);
}

// tcgen05 path: head_dim 64, Tp <= 384 (S row + O fit the 512 TMEM columns and the tiles fit shared memory); the tensor maps
// (Q: box 64 x min(128, Tp), K / V: box 64 x Tp or Tp / 2, all SWIZZLE_128B) are built by the plan with attention_tc_boxes().
bool attention_tc_supported(int T) {
    AttnTcParams p; size_t smem;
    return attn_tc_plan(T, 1, HD, 1, 0.125f, &p, &smem);
}
bool attention_tc_eligible(int T) {
    static const bool off = getenv("TMAE_NO_TC_ATTN") != nullptr;
    return !off && attention_tc_supported(T);
}
int attention_tc_tp(int T) { return attn_tp(T); }
// Which form of the kernel serves (T, H): lite (one softmax group, two CTAs per SM) for short rows while several streams
// share the GPU, else the full form; TMAE_ATTN_LITE=1 / 0 forces lite on / off (A/B runs).
// duo (two heads per 128-row tile at T = 65, cls queries on the tail warp) is OPT-IN (mode 3 / TMAE_ATTN_DUO=1): measured
// slower than the plain form on B200 (0.285 vs 0.227 ms for the 12 launches of the B-64 forward) - the softmax is
// issue-bound, so filling all four TMEM lane quarters doubles the per-item softmax time while the items halve, and the
// 56 KB stages leave a 2-deep pipeline.
static void attn_mode(int T, int H, int mode, bool* lite, bool* duo) {
    static const char* lite_env = getenv("TMAE_ATTN_LITE");
    static const bool duo_env = getenv("TMAE_ATTN_DUO") != nullptr;
    const bool share_sm = mode == 2;
    *duo = (mode == 3 || duo_env) && T == 65 && (H & 1) == 0;
    *lite = !*duo && attn_tp(T) <= 96 && (lite_env ? lite_env[0] == '1' : share_sm);
}
void attention_tc_boxes(int T, int H, int mode, int* q_rows, int* kv_rows) {
    AttnTcParams p = {}; size_t smem = 0;
    bool lite, duo;
    attn_mode(T, H, mode, &lite, &duo);
    attn_tc_plan(T, H, H * HD, 1, 0.125f, &p, &smem, lite, duo);
    *q_rows = p.qrows; *kv_rows = p.krows;
}
// host-only view of the plan (tests): out[12] = {supported, Tp, q_tiles, tail_rows, n_items, nbuf, nst, tmem_cols, smem_bytes,
// q_box_rows, kv_box_rows, form (0 full, 1 lite, 2 duo)}
bool attention_tc_describe(int T, int H, int N, int mode, int* out) {
    AttnTcParams p = {}; size_t smem = 0;
    bool lite, duo;
    attn_mode(T, H, mode, &lite, &duo);
    const bool ok = attn_tc_plan(T, H, H * HD, N, 0.125f, &p, &smem, lite, duo);
    out[0] = ok ? 1 : 0; out[1] = attn_tp(T); out[2] = p.q_tiles; out[3] = p.tail_rows; out[4] = p.n_items; out[5] = p.nbuf; out[6] = p.nst;
    out[7] = (int)p.tmem_cols; out[8] = (int)smem; out[9] = p.qrows; out[10] = p.krows; out[11] = duo ? 2 : (lite ? 1 : 0);
    return ok;
}
cudaError_t launch_attention_tc(const CUtensorMap* map_q, const CUtensorMap* map_kv, const __nv_bfloat16* qkv, __nv_bfloat16* out, int N,
                                int T, int H, int C, float scale, cudaStream_t st, long long* dbg, int mode) {
    if (C != H * HD) return cudaErrorInvalidValue;
    AttnTcParams p; size_t smem;
    bool lite, duo;
    attn_mode(T, H, mode, &lite, &duo);
    if (!attn_tc_plan(T, H, C, N, scale, &p, &smem, lite, duo)) return cudaErrorInvalidValue;
    p.dbg = dbg;
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    TMAE_CARVEOUT_ONCE((attention_tc_kernel<3, 2>));
    TMAE_CARVEOUT_ONCE((attention_tc_kernel<3, 1>));
    TMAE_CARVEOUT_ONCE((attention_tc_kernel<4, 2>));
    TMAE_CARVEOUT_ONCE((attention_tc_kernel<0, 2>));
    if (lite) {
        const int grid = p.n_items < 2 * sms ? p.n_items : 2 * sms;
        return launch_k(attention_tc_kernel<3, 1>, dim3(grid), dim3(192), smem, st, true, *map_q, *map_kv, qkv, out, p);
    }
    const int grid = p.n_items < sms ? p.n_items : sms;
    const dim3 blk(kAttnTcThreads + 32);          // + the tail warp
    if (p.duo) {
        TMAE_CARVEOUT_ONCE((attention_tc_kernel<3, 2, true>));
        static const cudaError_t cfg = cudaFuncSetAttribute(attention_tc_kernel<3, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (cfg != cudaSuccess) return cfg;
        return launch_k(attention_tc_kernel<3, 2, true>, dim3(grid), blk, smem, st, true, *map_q, *map_kv, qkv, out, p);
    }
    if (p.Tp <= 96) return launch_k(attention_tc_kernel<3, 2>, dim3(grid), blk, smem, st, true, *map_q, *map_kv, qkv, out, p);
    if (p.Tp <= 128) return launch_k(attention_tc_kernel<4, 2>, dim3(grid), blk, smem, st, true, *map_q, *map_kv, qkv, out, p);
    return launch_k(attention_tc_kernel<0, 2>, dim3(grid), blk, smem, st, true, *map_q, *map_kv, qkv, out, p);
}

cudaError_t launch_attention_f32(const __nv_bfloat16* qkv, long long qkv_lo, __nv_bfloat16* out, long long out_lo, int N,
                                 int T, int H, int C, float scale, cudaStream_t st) {
    if (C != H * HD || qkv_lo == 0 || out_lo == 0) return cudaErrorInvalidValue;
    if (attn_f32_smem(T) > 227 * 1024) return cudaErrorInvalidValue;
    TMAE_CARVEOUT_ONCE(attention_f32_kernel);
    return launch_k(attention_f32_kernel, dim3(N * H), dim3(32 * kAttnF32Warps), attn_f32_smem(T), st, true, qkv, qkv_lo, out,
                    out_lo, T, H, C, scale);
}

}  // namespace tmae
