// tcgen05 / TMEM / TMA GEMM engine for sm_100a.
//
// One CTA computes a 128 x block_n fp32 accumulator tile in tensor memory:
//   warp 0     : TMA producer - per pipeline stage one or two k-blocks (128x64 bf16 A tile + block_n x 64 bf16 weight
//                tile, 128B-swizzled); A = 2-D box of a token matrix (one map per concatenated channel segment), or a
//                4-D box of a compact image tensor for 3x3 convs, optionally one haloed box shared by three dy taps
//   warp 1     : allocates TMEM, issues tcgen05.mma (M=128, N=block_n, K=16) x 4 per k-block from one elected lane,
//                tcgen05.commit releases the smem stage / publishes the accumulator
//   warps 2-9  : epilogue - tcgen05.ld 32 lanes x 32 columns, + bias, GELU / 0.5*tanh, residual / pos-embed add,
//                row remap (stride-2 subsample, PixelShuffle, token rows), bf16 / fp32 stores or TMA stores;
//                warp 2 doubles as second TMA producer on narrow tiles
// Variants: persistent tile loop with double-buffered TMEM (gemm_tc_persistent_kernel), CUDA-core checker
// (gemm_simt_kernel).  Precise layers (split-bf16, three tensor-core terms per product) are the same kernels walking
// three times as many K segments (gemm.cuh).
// Serves reference layers: PatchEmbed conv (MCM.py:300-302), Block linears (MCM.py:313-322), g_a 1x1 convs
// (MCM.py:77-93), h_a / h_s / cc_transform / lrp_transform 3x3 convs (MCM.py:115-293).
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm.cuh"
#include "kernels.h"

namespace tmae {

// ---------------------------------------------------------------------------------------------------------
// epilogue shared by the tensor-core kernel and the CUDA-core checker
// ---------------------------------------------------------------------------------------------------------
// Register-resident copy of the epilogue description (the parameter block lives in global memory; the inline-asm
// "memory" clobbers of the tcgen05 wrappers would otherwise force every field to be re-read per use).
struct EpiCtx {
    const float* bias;
    const float* resid;
    const int64_t* gather_ids;
    OutSpec out[2];
    const void* out_map;
    const float* ln_stats_in;
    const float* ln_wsum;
    float* ln_stats_out;
    __nv_bfloat16* xbf_out;
    float ln_inv_c, ln_eps;
    int ln_chunks;
    int act, resid_ld, resid_map, M, N, in_mode, s, K, T, n_img, box_y, box_n, y_tiles, rows_used, exact_act;
    const GemmParams* gp;                  // the parameter block itself (EPI_GAUSS reads its gc_* fields)
};

__device__ __forceinline__ EpiCtx load_epi(const GemmParams& p) {
    EpiCtx e;
    e.bias = p.bias; e.resid = p.resid; e.gather_ids = p.gather_ids;
    e.out[0] = p.out[0]; e.out[1] = p.out[1];
    e.out_map = &p.out_map;
    e.act = p.act; e.resid_ld = p.resid_ld; e.resid_map = p.resid_map;
    e.M = p.M; e.N = p.N; e.in_mode = p.in_mode; e.s = p.s; e.K = p.K; e.T = p.T;
    e.n_img = p.n_img; e.box_y = p.box_y; e.box_n = p.box_n; e.y_tiles = p.y_tiles; e.rows_used = p.rows_used;
    e.exact_act = p.mma_terms > 1;
    e.ln_stats_in = p.ln_stats_in; e.ln_wsum = p.ln_wsum; e.ln_stats_out = p.ln_stats_out; e.xbf_out = p.xbf_out;
    e.ln_inv_c = p.ln_inv_c; e.ln_eps = p.ln_eps; e.ln_chunks = p.ln_chunks;
    e.gp = &p;
    return e;
}

// Conv tiles: CTA tile `m_tile` covers image rows [y0, y0 + box_y) of images [n0, n0 + box_n).
__device__ __forceinline__ void conv_tile_origin(int m_tile, int y_tiles, int box_y, int box_n, int& y0, int& n0) {
    const int nt = m_tile / y_tiles;
    y0 = (m_tile - nt * y_tiles) * box_y;
    n0 = nt * box_n;
}

struct RowCtx {
    int valid, n, y, x, lin;
};

// r = accumulator row (0..127) of CTA tile `m_tile`.  Linear row spaces: row m_tile*128 + r.  Conv: the A tile is the
// TMA box [x][nl][yl] flattened, r = (yl * box_n + nl) * s + x, and the row it stands for is pixel (n0+nl, y0+yl, x).
__device__ __forceinline__ RowCtx decode_row(const EpiCtx& p, int m_tile, int r) {
    RowCtx c;
    c.n = c.y = c.x = 0;
    if (p.in_mode == IN_CONV) {
        int y0, n0;
        conv_tile_origin(m_tile, p.y_tiles, p.box_y, p.box_n, y0, n0);
        const int per_y = p.s * p.box_n;
        const int yl = r / per_y, rem = r - yl * per_y;
        const int nl = rem / p.s;
        c.x = rem - nl * p.s;
        c.y = y0 + yl;
        c.n = n0 + nl;
        c.valid = (r < p.rows_used) && (c.n < p.n_img) && (c.y < p.s);
        c.lin = c.n * p.K + c.y * p.s + c.x;
    } else {
        c.lin = m_tile * kBlockM + r;
        c.valid = c.lin < p.M;
        if (p.in_mode == IN_COMPACT) {
            c.n = c.lin / p.K;
            const int j = c.lin - c.n * p.K;
            c.y = j / p.s;
            c.x = j - c.y * p.s;
        }
    }
    return c;
}

// q = PixelShuffle quadrant (dy*2+dx) of the column group; returns -1 when this row produces no output.
__device__ __forceinline__ long long map_row(const EpiCtx& p, int map, const RowCtx& r, int q) {
    if (!r.valid) return -1;
    switch (map) {
        case MAP_SAME: return r.lin;
        case MAP_TO_TOKEN: return (long long)r.n * p.T + 1 + r.y * p.s + r.x;
        case MAP_S2: {
            if ((r.y | r.x) & 1) return -1;
            const int s2 = p.s >> 1;
            return (long long)r.n * s2 * s2 + (r.y >> 1) * s2 + (r.x >> 1);
        }
        case MAP_SHUF: {
            const int s2 = p.s << 1;
            return (long long)r.n * s2 * s2 + (2 * r.y + (q >> 1)) * s2 + 2 * r.x + (q & 1);
        }
        case MAP_GATHER1: return p.gather_ids[r.lin] + 1;
    }
    return -1;
}

// erf-form GELU with erf from Abramowitz & Stegun 7.1.26 (|err| <= 1.5e-7): 2 MUFU + ~12 FMA instead of erff's ~40
// instructions; the result is rounded to bf16 (2^-9 relative) right after, so the approximation is invisible.
__device__ __forceinline__ float gelu_erf_fast(float x) {
    const float z = fabsf(x) * 0.70710678118654752440f;
    float t;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));      // 1 MUFU (1 ulp) instead of IEEE rcp
    float poly = fmaf(1.061405429f, t, -1.453152027f);
    poly = fmaf(poly, t, 1.421413741f);
    poly = fmaf(poly, t, -0.284496736f);
    poly = fmaf(poly, t, 0.254829592f);
    poly *= t;
    float ex;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex) : "f"(z * z * -1.4426950408889634f));    // exp(-z^2)
    const float half_x = 0.5f * x;
    // 0.5 x (1 + erf(x / sqrt 2)) = x/2 + |x/2| * erf(|z|)   (erf is odd, so the sign of x cancels)
    return fmaf(fabsf(half_x), fmaf(-poly, ex, 1.0f), half_x);
}

template <int ACT>
__device__ __forceinline__ float act_fast(float v) {
    if (ACT == ACT_GELU) return gelu_erf_fast(v);
    if (ACT == ACT_HALF_TANH) return 0.5f * tanhf(v);
    return v;
}

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == ACT_GELU) return gelu_erf(v);
    if (act == ACT_HALF_TANH) return 0.5f * tanhf(v);
    return v;
}

// Residual add + stores for `NV` (4 or 8) consecutive output channels of one row, rows already mapped.
template <int NV>
__device__ __forceinline__ void finish_store(const EpiCtx& p, float (&v)[NV], int ocol, long long rrow, long long orow0,
                                             long long orow1) {
    if (p.resid != nullptr && rrow >= 0) {
        const float* src = p.resid + rrow * p.resid_ld + ocol;
#pragma unroll
        for (int i = 0; i < NV; i += 4) {
            const float4 r4 = *reinterpret_cast<const float4*>(src + i);
            v[i] += r4.x; v[i + 1] += r4.y; v[i + 2] += r4.z; v[i + 3] += r4.w;
        }
    }
#pragma unroll
    for (int o = 0; o < 2; ++o) {
        const OutSpec& os = p.out[o];
        const long long orow = o == 0 ? orow0 : orow1;
        if (os.dtype == OUT_NONE || orow < 0) continue;
        if (os.dtype == OUT_BF16) {
            __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(os.ptr) + orow * os.ld + ocol;
            if (os.lo_off != 0) {
#pragma unroll
                for (int i = 0; i < NV; i += 4) store_bf16x4_planes(dst + i, os.lo_off, v[i], v[i + 1], v[i + 2], v[i + 3]);
            } else if (NV == 8) {
                uint4 pk;
                pk.x = pack_bf16x2(v[0], v[1]); pk.y = pack_bf16x2(v[2], v[3]);
                pk.z = pack_bf16x2(v[NV - 4], v[NV - 3]); pk.w = pack_bf16x2(v[NV - 2], v[NV - 1]);
                *reinterpret_cast<uint4*>(dst) = pk;
            } else {
                uint2 pk;
                pk.x = pack_bf16x2(v[0], v[1]); pk.y = pack_bf16x2(v[2], v[3]);
                *reinterpret_cast<uint2*>(dst) = pk;
            }
        } else {
            float* dst = reinterpret_cast<float*>(os.ptr) + orow * os.ld + ocol;
#pragma unroll
            for (int i = 0; i < NV; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
    }
}

// Store 4 consecutive channels of one mapped row (row < 0: nothing to write).
__device__ __forceinline__ void store_out4(const OutSpec& os, int orow, int ocol, const float (&v)[4]) {
    if (os.dtype == OUT_NONE || orow < 0) return;
    if (os.dtype == OUT_BF16) {
        __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(os.ptr) + (long long)orow * os.ld + ocol;
        store_bf16x4_planes(dst, os.lo_off, v[0], v[1], v[2], v[3]);
    } else {
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(os.ptr) + (long long)orow * os.ld + ocol) =
            make_float4(v[0], v[1], v[2], v[3]);
    }
}

// Row-per-thread variant (CUDA-core checker): finish 8 consecutive output channels [col, col+8) of one row.
__device__ __forceinline__ void epilogue8(const EpiCtx& p, const RowCtx& r, int col, float (&v)[8]) {
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col));
    const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col + 4));
    v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
    v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = apply_act(v[i], p.act);
    // PixelShuffle bookkeeping: weights are packed quadrant-major, so consecutive columns share (dy,dx).
    int q = 0, ocol = col;
    if (p.out[0].map == MAP_SHUF || p.out[1].map == MAP_SHUF) {
        const int cq = p.N >> 2;
        q = col / cq;
        ocol = col - q * cq;
    }
    const long long rrow = p.resid ? map_row(p, p.resid_map, r, q) : -1;
    finish_store<8>(p, v, ocol, rrow, map_row(p, p.out[0].map, r, q), map_row(p, p.out[1].map, r, q));
}

// ---------------------------------------------------------------------------------------------------------
// tensor-core kernel
// ---------------------------------------------------------------------------------------------------------
constexpr int kGemmThreads = 320;                     // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue
constexpr int kEpiPitch = 36;                         // floats per staged accumulator row (32 + 4 pad)
constexpr int kAStageBytes = kBlockM * kBlockK * 2;   // 16 KB

// EPI selects a compile-time specialisation of the store phase:
//   EPI_GENERIC        any row map / two outputs / gathered residual (patch embed, g_a.6, strided, PixelShuffle, mu/sigma, LRP)
//   EPI_BF16_SAME      one bf16 output at the accumulator's own row (QKV, fc1, g_a.0-4, every conv mid layer)
//   EPI_F32_SAME_RESID one fp32 output at the accumulator's own row with an fp32 residual at the same row (proj, fc2)
//   EPI_BF16_TMA       EPI_BF16_SAME when the tile is 128 consecutive output rows and block_n % 32 == 0: bias/activation in
//                      registers, bf16 boxes of 32 columns staged in smem (64B swizzle) and written by TMA stores
//   EPI_GAUSS          last layer of cc_transform_mean[i] + cc_transform_scale[i] as one block-diagonal 64-column GEMM: the
//                      Gaussian conditional (quantise, likelihood, symbols, indexes, y_hat, rate) runs here, thread = pixel
//   EPI_GAUSS_IDX      the same layer in the decoder (GemmParams::gc_on == 2): mu, sigma and scale-table indexes only
enum EpiKind : int { EPI_GENERIC = 0, EPI_BF16_SAME = 1, EPI_F32_SAME_RESID = 2, EPI_BF16_TMA = 3, EPI_GAUSS = 4, EPI_GAUSS_IDX = 5 };
constexpr uint32_t kStoreBoxBytes = kBlockM * 32 * 2;      // one 128 x 32 bf16 box

// ---------------------------------------------------------------------------------------------------------
// Epilogue of one 128 x block_n accumulator tile, executed by the 8 epilogue warps (warp index 2..9; TMEM lane
// quarter = warp % 4, two warps per quarter alternate 32-column chunks).
// Phase 1 (thread = accumulator row): TMEM -> registers -> smem staging tile (raw fp32 accumulators).
// Phase 2 (8 lanes = 32 consecutive channels of one row, 4 rows per instruction): + bias, activation, residual add,
// coalesced 64 / 128-byte row segments to global memory.
// ---------------------------------------------------------------------------------------------------------
template <int ACT, int EPI, bool EXACT>
__device__ __forceinline__ void epilogue_tile_impl(const EpiCtx& e, int m_tile, int n0, int block_n, uint32_t tmem_acc,
                                                   uint32_t stage_base, int warp, int lane, uint64_t* wait_bar,
                                                   uint32_t wait_parity, long long* ticks, int nsub) {
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;                  // which of the `nsub` warps of this TMEM lane quarter
    // precise layers evaluate GELU with erff (the fast form's 1.5e-7 absolute error is visible next to fp32-exact products);
    // a compile-time choice: a per-element runtime select cost the GELU layers 20 % (measured)
    auto act = [](float x) { return (ACT == ACT_GELU && EXACT) ? gelu_erf(x) : act_fast<ACT>(x); };
    const int cstride = 32 * nsub;
    const int m0 = m_tile * kBlockM;                   // first row of the tile in a linear row space
    if (EPI == EPI_BF16_TMA) {
        // Thread = accumulator row: TMEM -> registers, + bias, activation, pack to bf16, 4 x 16-byte swizzled smem stores
        // into a 128 x 32 box; the four warps that share a column subset (`half`) sync on a named barrier and one thread
        // hands the box to the TMA (which clips rows >= M and columns >= N).  Two boxes per subset are in flight.
        const int row = quarter * 32 + lane;
        const uint32_t row_off = (uint32_t)row * 64u, sw = (uint32_t)((row >> 1) & 3);
        const uint32_t buf0 = stage_base + (uint32_t)half * 2u * kStoreBoxBytes;
        const bool issuer = quarter == 0 && lane == 0;
        const int bar_id = 1 + half;
        const bool conv_t = e.in_mode == IN_CONV;                    // conv: the tile is a 4-D box (x, images, rows) of the output
        int ty0 = 0, tn0 = 0;
        if (conv_t) conv_tile_origin(m_tile, e.y_tiles, e.box_y, e.box_n, ty0, tn0);
        const int nboxes = block_n >> 5;
        // folded LayerNorm (see GemmParams::ln_stats_in): this thread's row statistics, fetched before the accumulator wait
        const bool fold = e.ln_stats_in != nullptr;
        float ln_mean = 0.f, ln_rstd = 1.f;
        if (fold && m0 + row < e.M) {
            // one (sum, sum of squares) partial per 32-column chunk of the row, written by the producing layer: summed in
            // a fixed order, so the statistics do not depend on tiling, batch size or run (no atomics)
            const float2* sp = reinterpret_cast<const float2*>(e.ln_stats_in) + (long long)(m0 + row) * e.ln_chunks;
            float s1 = 0.f, s2 = 0.f;
            for (int c = 0; c < e.ln_chunks; ++c) { const float2 v = sp[c]; s1 += v.x; s2 += v.y; }
            ln_mean = s1 * e.ln_inv_c;
            ln_rstd = rsqrtf(fmaxf(s2 * e.ln_inv_c - ln_mean * ln_mean, 0.f) + e.ln_eps);
        }
        const float ln_nm = -ln_mean;
        mbar_wait(wait_bar, wait_parity);
        tc_fence_after();
        if (ticks && warp == 2 && lane == 0) ticks[5] = globaltimer_ns();
        const uint32_t lane_base = tmem_acc + ((uint32_t)(quarter * 32) << 16);
        int it = 0;
        for (int b = half; b < nboxes; b += nsub, ++it) {
            const int c0 = b * 32;
            uint32_t acc[32];
            tmem_ld_32x32b_x32(lane_base + (uint32_t)c0, acc);
            tmem_ld_wait();
            uint32_t pk[16];
#pragma unroll
            for (int g4 = 0; g4 < 8; ++g4) {
                const int col = n0 + c0 + g4 * 4;
                const float4 bb = col < e.N ? __ldg(reinterpret_cast<const float4*>(e.bias + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
                float a0 = __uint_as_float(acc[g4 * 4]), a1 = __uint_as_float(acc[g4 * 4 + 1]);
                float a2 = __uint_as_float(acc[g4 * 4 + 2]), a3 = __uint_as_float(acc[g4 * 4 + 3]);
                if (fold) {                                  // rstd * (acc - mean * wsum) + bias'
                    const float4 ws = col < e.N ? __ldg(reinterpret_cast<const float4*>(e.ln_wsum + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    a0 = fmaf(ln_nm, ws.x, a0) * ln_rstd; a1 = fmaf(ln_nm, ws.y, a1) * ln_rstd;
                    a2 = fmaf(ln_nm, ws.z, a2) * ln_rstd; a3 = fmaf(ln_nm, ws.w, a3) * ln_rstd;
                }
                pk[g4 * 2] = pack_bf16x2(act(a0 + bb.x), act(a1 + bb.y));
                pk[g4 * 2 + 1] = pack_bf16x2(act(a2 + bb.z), act(a3 + bb.w));
            }
            const uint32_t buf = buf0 + (uint32_t)(it & 1) * kStoreBoxBytes;
            if (it >= 2) {                                 // the store that last read this buffer must be done with it
                if (issuer) bulk_wait_group_read<1>();
                named_bar_sync(bar_id, 128);
            }
#pragma unroll
            for (int ch = 0; ch < 4; ++ch)
                sts128(buf + row_off + ((((uint32_t)ch) ^ sw) << 4), pk[ch * 4], pk[ch * 4 + 1], pk[ch * 4 + 2], pk[ch * 4 + 3]);
            fence_proxy_async_smem();                      // generic-proxy writes -> visible to the TMA (async proxy)
            named_bar_sync(bar_id, 128);
            if (issuer) {
                if (conv_t) tma_store_4d_a(e.out_map, buf, n0 + c0, 0, tn0, ty0);
                else tma_store_2d_a(e.out_map, buf, n0 + c0, m0);
                bulk_commit_group();
            }
        }
        if (issuer) bulk_wait_group_read<0>();             // smem may be reused / released once the TMA has read it
        return;
    }
    if (EPI == EPI_GAUSS) {
        // Columns are interleaved by the weight pack: 32-column chunk b = [mu of channels 16 b .. 16 b + 15 | sigma of the same
        // channels], so the CTA that owns chunk b (block_n = 32) holds both statistics of its 16 channels of every pixel of
        // the tile (MCM.py:762-776).
        const GemmParams& g = *e.gp;
        const IoBlock* io = reinterpret_cast<const IoBlock*>(g.gc_io);
        float* lik_out = io->out.y_likelihoods;
        int32_t* sym_out = io->out.y_symbols;
        int16_t* sym16_out = io->out.y_symbols_i16;
        int32_t* idx_out = io->out.y_indexes;
        const RowCtx r = decode_row(e, m_tile, quarter * 32 + lane);
        mbar_wait(wait_bar, wait_parity);
        tc_fence_after();
        const uint32_t lane_base = tmem_acc + ((uint32_t)(quarter * 32) << 16);
        float lg = 0.f;
        {
            // block_n == 32: this CTA owns chunk b = n0 / 32, i.e. channels [16 b, 16 b + 16); the two warps of a TMEM lane
            // quarter take 8 channels each (2 x 32 CTAs x 8 warps share the erfc / log2 work of a slice)
            const int b = n0 >> 5;
            uint32_t acc[32];
            tmem_ld_32x32b_x32(lane_base, acc);
            tmem_ld_wait();
            if (r.valid) {
                const int c0 = g.gc_col0 + b * 16;
                const size_t off = (size_t)r.lin * g.gc_ld + c0;
#pragma unroll
                for (int jj = 0; jj < 2; ++jj) {
                    const int j = half * 2 + jj;                     // 4-channel group of the chunk
                    const float4 yv = *reinterpret_cast<const float4*>(g.gc_y + off + 4 * j);
                    const float4 bm = __ldg(reinterpret_cast<const float4*>(e.bias + n0 + 4 * j));
                    const float4 bs = __ldg(reinterpret_cast<const float4*>(e.bias + n0 + 16 + 4 * j));
                    float a[8];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {                    // dynamic j: select the registers without local memory
                        a[q] = __uint_as_float(half == 0 ? acc[4 * jj + q] : acc[8 + 4 * jj + q]);
                        a[4 + q] = __uint_as_float(half == 0 ? acc[16 + 4 * jj + q] : acc[24 + 4 * jj + q]);
                    }
                    const float4 mv = make_float4(a[0] + bm.x, a[1] + bm.y, a[2] + bm.z, a[3] + bm.w);
                    const float4 sv = make_float4(a[4] + bs.x, a[5] + bs.y, a[6] + bs.z, a[7] + bs.w);
                    float4 lk, sy, yh;
                    gaussian_elem(yv.x, mv.x, sv.x, lk.x, sy.x, yh.x);
                    gaussian_elem(yv.y, mv.y, sv.y, lk.y, sy.y, yh.y);
                    gaussian_elem(yv.z, mv.z, sv.z, lk.z, sy.z, yh.z);
                    gaussian_elem(yv.w, mv.w, sv.w, lk.w, sy.w, yh.w);
                    const size_t o4 = off + 4 * j;
                    *reinterpret_cast<float4*>(g.gc_mu + o4) = mv;
                    *reinterpret_cast<float4*>(g.gc_sigma + o4) = sv;
                    *reinterpret_cast<float4*>(g.gc_yhat + o4) = yh;
                    store_bf16x4_planes(g.gc_yhat_bf + o4, g.gc_yhat_lo, yh.x, yh.y, yh.z, yh.w);
                    if (lik_out) *reinterpret_cast<float4*>(lik_out + o4) = lk;
                    if (sym_out) *reinterpret_cast<int4*>(sym_out + o4) = make_int4((int)sy.x, (int)sy.y, (int)sy.z, (int)sy.w);
                    if (sym16_out) {
                        auto sat = [](float v) { return (int16_t)fminf(fmaxf(v, -32768.f), 32767.f); };
                        short4 s4v;
                        s4v.x = sat(sy.x); s4v.y = sat(sy.y); s4v.z = sat(sy.z); s4v.w = sat(sy.w);
                        *reinterpret_cast<short4*>(sym16_out + o4) = s4v;
                    }
                    if (idx_out && g.gc_table)              // GaussianConditional.build_indexes (MCM.py:839)
                        *reinterpret_cast<int4*>(idx_out + o4) = scale_indexes4(g.gc_table, g.gc_ntable, sv);
                    lg += (log2f(lk.x) + log2f(lk.y)) + (log2f(lk.z) + log2f(lk.w));
                }
            }
        }
        // rate: sum of log2 likelihoods per image (fp32 per warp when its 32 pixels belong to one image, fp64 atomics per image)
        const unsigned vm = __ballot_sync(0xffffffffu, r.valid != 0);
        if (vm != 0u) {
            const int n_first = __shfl_sync(0xffffffffu, r.n, __ffs(vm) - 1);
            const bool same = __all_sync(0xffffffffu, !r.valid || r.n == n_first);
            if (same) {
                const float sm = warp_sum(r.valid ? lg : 0.f);
                if (lane == 0 && sm != 0.f) atomicAdd(g.gc_rate + n_first, (double)sm);
            } else if (r.valid) {
                atomicAdd(g.gc_rate + r.n, (double)lg);
            }
        }
        return;
    }
    if (EPI == EPI_GAUSS_IDX) {
        // Decoder side of EPI_GAUSS: same column interleave and bias adds, but no y exists yet - the store phase writes mu,
        // sigma and the scale-table indexes the range decoder needs before it can produce the slice's symbols.  Indexes go
        // out in the range coder's order: per image, channel-major (c, y, x).
        const GemmParams& g = *e.gp;
        const IoBlock* io = reinterpret_cast<const IoBlock*>(g.gc_io);
        int32_t* idx_out = io->out.y_indexes;
        const RowCtx r = decode_row(e, m_tile, quarter * 32 + lane);
        mbar_wait(wait_bar, wait_parity);
        tc_fence_after();
        const uint32_t lane_base = tmem_acc + ((uint32_t)(quarter * 32) << 16);
        const int b = n0 >> 5;
        uint32_t acc[32];
        tmem_ld_32x32b_x32(lane_base, acc);
        tmem_ld_wait();
        if (r.valid) {
            const int c0 = g.gc_col0 + b * 16;
            const size_t off = (size_t)r.lin * g.gc_ld + c0;
            int32_t* idx_px = idx_out + (size_t)r.n * g.gc_ld * g.gc_pixels + (r.y * e.s + r.x);
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
                const int j = half * 2 + jj;
                const float4 bm = __ldg(reinterpret_cast<const float4*>(e.bias + n0 + 4 * j));
                const float4 bs = __ldg(reinterpret_cast<const float4*>(e.bias + n0 + 16 + 4 * j));
                float a[8];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    a[q] = __uint_as_float(half == 0 ? acc[4 * jj + q] : acc[8 + 4 * jj + q]);
                    a[4 + q] = __uint_as_float(half == 0 ? acc[16 + 4 * jj + q] : acc[24 + 4 * jj + q]);
                }
                const float4 mv = make_float4(a[0] + bm.x, a[1] + bm.y, a[2] + bm.z, a[3] + bm.w);
                const float4 sv = make_float4(a[4] + bs.x, a[5] + bs.y, a[6] + bs.z, a[7] + bs.w);
                const size_t o4 = off + 4 * j;
                *reinterpret_cast<float4*>(g.gc_mu + o4) = mv;
                *reinterpret_cast<float4*>(g.gc_sigma + o4) = sv;
                const int4 id = scale_indexes4(g.gc_table, g.gc_ntable, sv);
                int32_t* dst = idx_px + (size_t)(c0 + 4 * j) * g.gc_pixels;
                dst[0] = id.x;
                dst[g.gc_pixels] = id.y;
                dst[2 * g.gc_pixels] = id.z;
                dst[3 * g.gc_pixels] = id.w;
            }
        }
        return;
    }
    const RowCtx r = decode_row(e, m_tile, quarter * 32 + lane);
    const bool conv = e.in_mode == IN_CONV;            // conv tiles: output rows come from the decoded pixel, not m0 + r
    const bool shuf = e.out[0].map == MAP_SHUF || e.out[1].map == MAP_SHUF;
    const int cq = e.N >> 2;
    const uint32_t stage_a = stage_base + (uint32_t)(warp - 2) * 32u * kEpiPitch * 4u;   // this warp's staging tile
    const int rsub = lane >> 3, c4 = (lane & 7) * 4;
    // mapped rows of THIS thread's accumulator row (quadrant-dependent ones are refreshed per chunk)
    int my_rrow = e.resid ? (int)map_row(e, e.resid_map, r, 0) : -1;
    int my_orow0 = e.out[0].dtype != OUT_NONE ? (int)map_row(e, e.out[0].map, r, 0) : -1;
    int my_orow1 = e.out[1].dtype != OUT_NONE ? (int)map_row(e, e.out[1].map, r, 0) : -1;
    // bias of this lane's 4 channels for each of its (up to 4) column chunks: fetched before the accumulator wait
    auto load_bias = [&](int c0) {
        const int col = n0 + c0 + c4;
        return (c0 + c4 < block_n && col < e.N) ? __ldg(reinterpret_cast<const float4*>(e.bias + col))
                                                : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    float4 bias_next = load_bias(half * 32);
    const bool has_resid = e.resid != nullptr;
    const long long lo_off = e.out[0].lo_off;          // EPI_BF16_SAME of a layer that feeds a precise layer: second plane
    const unsigned valid_mask = __ballot_sync(0xffffffffu, r.valid != 0);   // rows of this quarter that produce output
    mbar_wait(wait_bar, wait_parity);
    tc_fence_after();
    if (ticks && warp == 2 && lane == 0) ticks[5] = globaltimer_ns();
    const uint32_t lane_base = tmem_acc + ((uint32_t)(quarter * 32) << 16);
    for (int c0 = half * 32; c0 < block_n; c0 += cstride) {
        const float4 b4 = bias_next;
        bias_next = load_bias(c0 + cstride);                        // prefetch for the next chunk of this warp
        uint32_t acc[32];
        if (block_n - c0 >= 32) {
            tmem_ld_32x32b_x32(lane_base + (uint32_t)c0, acc);
        } else {                                  // block_n is a multiple of 16
            uint32_t a16[16];
            tmem_ld_32x32b_x16(lane_base + (uint32_t)c0, a16);
#pragma unroll
            for (int i = 0; i < 16; ++i) { acc[i] = a16[i]; acc[16 + i] = 0u; }
        }
        tmem_ld_wait();
        if (ticks && warp == 2 && lane == 0 && c0 == half * 32) ticks[8] = globaltimer_ns();
#pragma unroll
        for (int g4 = 0; g4 < 8; ++g4)
            sts128(stage_a + (uint32_t)(lane * kEpiPitch + g4 * 4) * 4u, acc[g4 * 4], acc[g4 * 4 + 1], acc[g4 * 4 + 2],
                   acc[g4 * 4 + 3]);
        const int colbase = n0 + c0;
        int q = 0;
        if (shuf) {                                               // cq % 32 == 0 for PixelShuffle layers
            q = colbase / cq;
            my_orow0 = e.out[0].dtype != OUT_NONE ? (int)map_row(e, e.out[0].map, r, q) : -1;
            my_orow1 = e.out[1].dtype != OUT_NONE ? (int)map_row(e, e.out[1].map, r, q) : -1;
        }
        __syncwarp();
        if (ticks && warp == 2 && lane == 0 && c0 == half * 32) ticks[9] = globaltimer_ns();
        const int col = colbase + c4;
        const bool col_ok = col < e.N && c0 + c4 < block_n;
        const int ocol = col - q * (shuf ? cq : 0);
        if (EPI == EPI_BF16_SAME && conv) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int rr = it * 4 + rsub;
                const int orow = __shfl_sync(0xffffffffu, r.lin, rr);
                if (col_ok && ((valid_mask >> rr) & 1u)) {
                    const float4 t4 = lds128(stage_a + (uint32_t)(rr * kEpiPitch + c4) * 4u);
                    const float v0 = act(t4.x + b4.x), v1 = act(t4.y + b4.y);
                    const float v2 = act(t4.z + b4.z), v3 = act(t4.w + b4.w);
                    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(e.out[0].ptr) + (long long)orow * e.out[0].ld + col;
                    store_bf16x4_planes(dst, lo_off, v0, v1, v2, v3);
                }
            }
            __syncwarp();
            continue;
        }
        if (EPI == EPI_BF16_SAME) {
            if (col_ok) {
                __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(e.out[0].ptr) +
                                     (long long)(m0 + quarter * 32 + rsub) * e.out[0].ld + col;
                const long long step = 4ll * e.out[0].ld;
#pragma unroll
                for (int it = 0; it < 8; ++it, dst += step) {
                    const int rr = it * 4 + rsub;
                    if ((valid_mask >> rr) & 1u) {
                        const float4 t4 = lds128(stage_a + (uint32_t)(rr * kEpiPitch + c4) * 4u);
                        const float v0 = act(t4.x + b4.x), v1 = act(t4.y + b4.y);
                        const float v2 = act(t4.z + b4.z), v3 = act(t4.w + b4.w);
                        store_bf16x4_planes(dst, lo_off, v0, v1, v2, v3);
                    }
                }
            }
            __syncwarp();
            continue;
        }
        if (EPI == EPI_F32_SAME_RESID) {
            const int row0 = m0 + quarter * 32 + rsub;
            const long long step = 4ll * e.out[0].ld;
            float* dst = reinterpret_cast<float*>(e.out[0].ptr) + (long long)row0 * e.out[0].ld + col;
            const float* src = e.resid + (long long)row0 * e.resid_ld + col;
            const long long rstep = 4ll * e.resid_ld;
            const bool ln_out = e.ln_stats_out != nullptr;           // uniform: this layer feeds a folded LayerNorm
#pragma unroll
            for (int hb = 0; hb < 2; ++hb) {
                float4 rs[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rr = (hb * 4 + j) * 4 + rsub;
                    rs[j] = (col_ok && ((valid_mask >> rr) & 1u)) ? *reinterpret_cast<const float4*>(src + (hb * 4 + j) * rstep)
                                                                 : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rr = (hb * 4 + j) * 4 + rsub;
                    const bool ok = col_ok && ((valid_mask >> rr) & 1u);
                    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ok) {
                        const float4 t4 = lds128(stage_a + (uint32_t)(rr * kEpiPitch + c4) * 4u);
                        o = make_float4(act(t4.x + b4.x) + rs[j].x, act(t4.y + b4.y) + rs[j].y,
                                        act(t4.z + b4.z) + rs[j].z, act(t4.w + b4.w) + rs[j].w);
                        *reinterpret_cast<float4*>(dst + (hb * 4 + j) * step) = o;
                        if (e.xbf_out != nullptr) {                  // bf16 copy of the residual stream: A operand of the next GEMM
                            uint2 pk;
                            pk.x = pack_bf16x2(o.x, o.y);
                            pk.y = pack_bf16x2(o.z, o.w);
                            *reinterpret_cast<uint2*>(e.xbf_out + (long long)(row0 + (hb * 4 + j) * 4) * e.N + col) = pk;
                        }
                    }
                    if (ln_out) {                                    // (sum v, sum v^2) of this 32-column segment of the row
                        float s1 = (o.x + o.y) + (o.z + o.w);
                        float s2 = fmaf(o.x, o.x, o.y * o.y) + fmaf(o.z, o.z, o.w * o.w);
#pragma unroll
                        for (int sh = 1; sh < 8; sh <<= 1) {
                            s1 += __shfl_xor_sync(0xffffffffu, s1, sh);
                            s2 += __shfl_xor_sync(0xffffffffu, s2, sh);
                        }
                        if ((lane & 7) == 0 && ((valid_mask >> rr) & 1u) && col < e.N)       // this chunk's slot of the row
                            reinterpret_cast<float2*>(e.ln_stats_out)[(long long)(row0 + (hb * 4 + j) * 4) * (e.N >> 5) + (col >> 5)] =
                                make_float2(s1, s2);
                    }
                }
            }
            __syncwarp();
            continue;
        }
#pragma unroll
        for (int hb = 0; hb < 2; ++hb) {                          // two batches of 4 row-groups: loads first, then math
            int rrow[4], orow0[4], orow1[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int rr = (hb * 4 + j) * 4 + rsub;
                rrow[j] = __shfl_sync(0xffffffffu, my_rrow, rr);
                orow0[j] = __shfl_sync(0xffffffffu, my_orow0, rr);
                orow1[j] = __shfl_sync(0xffffffffu, my_orow1, rr);
            }
            if (col_ok) {
                float4 rs[4], t4[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    rs[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (has_resid)                                 // clamped row: always a valid address
                        rs[j] = *reinterpret_cast<const float4*>(e.resid + (long long)max(rrow[j], 0) * e.resid_ld + ocol);
                    t4[j] = lds128(stage_a + (uint32_t)(((hb * 4 + j) * 4 + rsub) * kEpiPitch + c4) * 4u);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float v[4];
                    v[0] = act(t4[j].x + b4.x) + rs[j].x;
                    v[1] = act(t4[j].y + b4.y) + rs[j].y;
                    v[2] = act(t4[j].z + b4.z) + rs[j].z;
                    v[3] = act(t4[j].w + b4.w) + rs[j].w;
                    store_out4(e.out[0], orow0[j], ocol, v);
                    store_out4(e.out[1], orow1[j], ocol, v);
                }
            }
            if (ticks && warp == 2 && lane == 0 && c0 == half * 32) ticks[10 + hb] = globaltimer_ns();
        }
        __syncwarp();
    }
}

template <int ACT, int EPI>
__device__ __forceinline__ void epilogue_tile(const EpiCtx& e, int m_tile, int n0, int block_n, uint32_t tmem_acc,
                                              uint32_t stage_base, int warp, int lane, uint64_t* wait_bar,
                                              uint32_t wait_parity, long long* ticks, int nsub = 2) {
    if (ACT == ACT_GELU && e.exact_act != 0)
        epilogue_tile_impl<ACT, EPI, true>(e, m_tile, n0, block_n, tmem_acc, stage_base, warp, lane, wait_bar, wait_parity, ticks, nsub);
    else
        epilogue_tile_impl<ACT, EPI, false>(e, m_tile, n0, block_n, tmem_acc, stage_base, warp, lane, wait_bar, wait_parity, ticks, nsub);
}

// ---------------------------------------------------------------------------------------------------------
// Pipeline stage = `kgroup` consecutive k-blocks (1, 2 or 4) behind ONE full / empty barrier pair:
//   [A atom 0 .. A atom G-1][B atom 0 .. B atom G-1],  A atom = 128 rows x 128 B, B atom = block_n rows x 128 B.
// Why: one producer <-> MMA handshake (wait, expect_tx / commit, wait) costs ~270-300 cycles per stage no matter how
// many stages there are (scripts/ubench_sync.cu: 2..16 stages, blocking or probing waits, acquire or relaxed), while the
// four MMAs of a k-block take 128 x block_n / 64 cycles: below block_n ~ 128 the handshake, not the tensor pipe, set the
// pace.  Grouping k-blocks divides the handshakes per k-block by G at the same number of bytes in flight.
// ---------------------------------------------------------------------------------------------------------

// TMA producer of one CTA tile (called by a whole warp; WARP-UNIFORM: all 32 lanes run the loop on identical values and
// only the TMA instructions are elect-predicated, so addresses and descriptors stay in uniform registers).
// Linear row spaces: A atom = 2-D box [64 ch, 128 rows].  Conv: 4-D box [64 ch, s, box_n, box_y] at pixel offset (dx, dy)
// of the tap; TMA zero-fills whatever falls outside the image (and images >= n_img), which IS the conv's zero padding.
// The pipeline position (stage / phase / stage_off) is carried across tiles by the caller.
__device__ __forceinline__ void produce_tile(const GemmParams& p, int m_tile, int n0, int total_kb, int stages, int kgroup,
                                             int stage_bytes, uint32_t pipe_base, uint32_t full_a, uint32_t empty_a,
                                             int& stage, uint32_t& phase, uint32_t& stage_off, long long* ticks,
                                             int prod_id = 0, int num_prod = 1, int pair = 0, uint32_t pair_rank = 0,
                                             uint32_t full_sig = 0) {
    // pair != 0 (CTA-pair launches, gemm_tc_pair_kernel): this CTA stages its own A tile and HALF of the weight tile (rows
    // [n0 + rank * block_n / 2, ...)); every load signals the LEADER's full barrier (`full_sig`, a shared::cluster
    // address) and only the leader arms it - with the bytes of both CTAs.
    // num_prod producer warps share the stage sequence round-robin (prod_id = which one this is): every producer walks
    // all stages (same coordinate / parity bookkeeping) but waits, arms and loads only its own.  One warp needs
    // ~300 cycles of barrier handshake PLUS ~140 cycles per 16 KB load it issues for every stage (the two add up: the
    // loop was producer bound at ~210 ns per k-block on the narrow conv tiles); two warps overlap each other's handshake.
    const int nseg = p.num_segs;
    const void* mapb = pair ? &p.b_map_pair : &p.b_map;
    const int b_rows = pair ? (p.block_n >> 1) : p.block_n;
    const int b_row0 = n0 + (pair ? (int)pair_rank * b_rows : 0);
    if (!pair) full_sig = full_a;
    const uint32_t tx_mult = pair ? 2u : 1u;
    const bool arm = !pair || pair_rank == 0;
    const int b_kb_per_tap = p.b_kb_per_tap;               // k-blocks per tap of the packed weights
    const bool conv = p.in_mode == IN_CONV;
    int y0 = 0, img0 = 0;
    if (conv) conv_tile_origin(m_tile, p.y_tiles, p.box_y, p.box_n, y0, img0);
    const int row = m_tile * kBlockM;
    const uint32_t b_atom = (uint32_t)(b_rows * kBlockK * 2);
    const uint32_t kb_bytes = (uint32_t)((conv ? p.rows_used : kBlockM) * kBlockK * 2) + b_atom;
    auto ld2d = [pair](uint32_t dst, const void* map, uint32_t bar, int c0, int c1) {
        if (pair) tma_load_2d_pair(dst, map, bar, c0, c1); else tma_load_2d_a(dst, map, bar, c0, c1);
    };
    auto ld4d = [pair](uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3) {
        if (pair) tma_load_4d_pair(dst, map, bar, c0, c1, c2, c3); else tma_load_4d_a(dst, map, bar, c0, c1, c2, c3);
    };
    const uint32_t b_base = (uint32_t)(kgroup * kAStageBytes);
    int sg = 0, k = 0, skb_cur = p.seg_kblocks[0];
    int koff = p.seg_b_kb0[0];                             // k-block of (sg, k) inside one tap of the packed weights
    int dx = -1;                                           // x-shift of the current taps (the weights are packed tap-major in (kh, kw) order)
    const void* map_cur = &p.a_map[0];
    int turn = 0;
    if (conv && p.conv_reuse) {
        // stage = one haloed A box (channel block k of segment sg at x-shift dx, rows y0-1 .. y0+box_y) + the B atoms of
        // the three taps (dy = -1, 0, +1) of that dx and channel block
        const uint32_t a_bytes = (uint32_t)(p.a_halo_rows * kBlockK * 2);
        const int n_stage = total_kb / 3;
        for (int it = 0; it < n_stage; ++it) {
            const bool mine = turn == prod_id;
            if (++turn == num_prod) turn = 0;
            if (mine) {
                mbar_wait_a(empty_a + 8u * stage, phase ^ 1u);
                if (elect_one()) {
                    const uint32_t fb = full_sig + 8u * stage;
                    if (arm) mbar_arrive_expect_tx_a(full_a + 8u * stage, tx_mult * (a_bytes + 3u * b_atom));
                    ld4d(pipe_base + stage_off, map_cur, fb, k * kBlockK, dx, img0, y0 - 1);
#pragma unroll
                    for (int t3 = 0; t3 < 3; ++t3)         // tap (dy = t3 - 1, dx): index t3 * 3 + (dx + 1) in (kh, kw) order
                        ld2d(pipe_base + stage_off + a_bytes + (uint32_t)t3 * b_atom, mapb, fb,
                             ((t3 * 3 + dx + 1) * b_kb_per_tap + koff) * kBlockK, b_row0);
                    if (ticks && it == 0) ticks[2] = globaltimer_ns();
                }
                __syncwarp();
            }
            ++koff;
            if (++k == skb_cur) {
                k = 0;
                if (++sg == nseg) { sg = 0; ++dx; }
                skb_cur = p.seg_kblocks[sg];
                koff = p.seg_b_kb0[sg];
                map_cur = &p.a_map[sg];
            }
            stage_off += (uint32_t)stage_bytes;
            if (++stage == stages) { stage = 0; phase ^= 1u; stage_off = 0; }
        }
        return;
    }
    // Per-k-block loads.  Conv k-blocks run in the SAME order as the conv_reuse path - dx, channel segment, channel block,
    // dy - so that a layer accumulates identically whichever path a launch takes (results do not depend on the batch size).
    int t3 = 0;
    for (int kb = 0; kb < total_kb;) {
        const int nk = min(kgroup, total_kb - kb);
        const bool mine = turn == prod_id;
        if (++turn == num_prod) turn = 0;
        const uint32_t fb = full_sig + 8u * stage;
        if (mine) {
            mbar_wait_a(empty_a + 8u * stage, phase ^ 1u);
            if (arm && elect_one()) mbar_arrive_expect_tx_a(full_a + 8u * stage, tx_mult * kb_bytes * (uint32_t)nk);
            __syncwarp();
        }
        for (int j = 0; j < nk; ++j, ++kb) {
            if (mine && elect_one()) {
                const uint32_t a_dst = pipe_base + stage_off + (uint32_t)(j * kAStageBytes);
                const uint32_t b_dst = pipe_base + stage_off + b_base + (uint32_t)j * b_atom;
                if (conv) {
                    ld4d(a_dst, map_cur, fb, k * kBlockK, dx, img0, y0 + t3 - 1);
                    ld2d(b_dst, mapb, fb, ((t3 * 3 + dx + 1) * b_kb_per_tap + koff) * kBlockK, b_row0);
                } else {
                    ld2d(a_dst, map_cur, fb, k * kBlockK, row);
                    ld2d(b_dst, mapb, fb, koff * kBlockK, b_row0);
                }
                if (ticks && kb == 0) ticks[2] = globaltimer_ns();
            }
            __syncwarp();
            if (conv && ++t3 < 3) continue;            // next dy tap of the same (dx, channel block)
            t3 = 0;
            ++koff;
            if (++k == skb_cur) {
                k = 0;
                if (++sg == nseg) { sg = 0; ++dx; }
                skb_cur = p.seg_kblocks[sg];
                koff = p.seg_b_kb0[sg];
                map_cur = &p.a_map[sg];
            }
        }
        stage_off += (uint32_t)stage_bytes;
        if (++stage == stages) { stage = 0; phase ^= 1u; stage_off = 0; }
    }
}

// MMA issuer of one CTA tile (whole warp, warp-uniform like the producer): accumulates total_kb k-blocks into
// tmem_acc, frees each pipeline stage with a tcgen05.commit and finally commits to `done_bar` (accumulator complete).
__device__ __forceinline__ void mma_tile(int block_n, int total_kb, int stages, int kgroup, int stage_bytes,
                                         uint32_t pipe_base, uint32_t full_a, uint32_t empty_a, uint32_t tmem_acc,
                                         uint32_t done_bar, int& stage, uint32_t& phase, uint32_t& stage_off,
                                         long long* ticks, int tick_issue, int tick_done,
                                         uint32_t reuse_a_bytes = 0, uint32_t reuse_dy_bytes = 0, int pair = 0) {
    // pair != 0: cta_group::2 MMAs of M = 256 over this CTA's and the peer's shared memory (each holds half of the B rows);
    // commits are multicast to the barriers at the same offsets in both CTAs
    const uint32_t idesc = umma_idesc_bf16_f32(pair ? 2 * kBlockM : kBlockM, block_n);
    const uint64_t desc0 = umma_smem_desc_sw128(pipe_base);       // + (byte offset >> 4) selects stage / atom / k-slice
    const uint32_t b_atom = (uint32_t)((pair ? (block_n >> 1) : block_n) * kBlockK * 2);
    auto mma = [pair](uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) {
        if (pair) umma_bf16_pair(d, a, b, id, acc); else umma_bf16(d, a, b, id, acc);
    };
    auto commit = [pair](uint32_t bar) { if (pair) umma_commit_pair(bar, (uint16_t)3); else umma_commit_a(bar); };
    if (reuse_a_bytes != 0) {
        // conv_reuse: total_kb counts k-blocks (9 taps); a stage holds the three dy taps of one (channel block, dx):
        // tap dy reads the haloed A box from row offset (dy + 1) * box_n * s (a whole number of 8-row swizzle atoms)
        const int n_stage = total_kb / 3;
        for (int it = 0; it < n_stage; ++it) {
            mbar_wait_a(full_a + 8u * stage, phase);
            tc_fence_after();
            if (elect_one()) {
                if (ticks && it == 0 && tick_issue >= 0) ticks[tick_issue] = globaltimer_ns();
#pragma unroll
                for (int t3 = 0; t3 < 3; ++t3) {
                    const uint64_t a_desc = desc0 + (uint64_t)((stage_off + (uint32_t)t3 * reuse_dy_bytes) >> 4);
                    const uint64_t b_desc = desc0 + (uint64_t)((stage_off + reuse_a_bytes + (uint32_t)t3 * b_atom) >> 4);
#pragma unroll
                    for (int k = 0; k < kBlockK / 16; ++k)
                        mma(tmem_acc, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (it | t3 | k) != 0 ? 1u : 0u);
                }
                commit(empty_a + 8u * stage);
                if (it == n_stage - 1) {
                    commit(done_bar);
                    if (ticks && tick_done >= 0) ticks[tick_done] = globaltimer_ns();
                }
            }
            __syncwarp();
            stage_off += (uint32_t)stage_bytes;
            if (++stage == stages) { stage = 0; phase ^= 1u; stage_off = 0; }
        }
        return;
    }
    const uint32_t b_base = (uint32_t)(kgroup * kAStageBytes);
    for (int kb = 0; kb < total_kb;) {
        const int nk = min(kgroup, total_kb - kb);
        mbar_wait_a(full_a + 8u * stage, phase);
        tc_fence_after();
        if (elect_one()) {
            if (ticks && kb == 0 && tick_issue >= 0) ticks[tick_issue] = globaltimer_ns();
            for (int j = 0; j < nk; ++j) {
                const uint64_t a_desc = desc0 + (uint64_t)((stage_off + (uint32_t)(j * kAStageBytes)) >> 4);
                const uint64_t b_desc = desc0 + (uint64_t)((stage_off + b_base + (uint32_t)j * b_atom) >> 4);
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k) {
                    // advance 16 bf16 = 32 B inside the 128B swizzle atom: +2 in the (addr >> 4) field
                    mma(tmem_acc, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, ((kb + j) | k) != 0 ? 1u : 0u);
                }
            }
            commit(empty_a + 8u * stage);                 // smem stage reusable once these MMAs retire
            if (kb + nk == total_kb) {
                commit(done_bar);                         // accumulator complete
                if (ticks && tick_done >= 0) ticks[tick_done] = globaltimer_ns();
            }
        }
        __syncwarp();
        kb += nk;
        stage_off += (uint32_t)stage_bytes;
        if (++stage == stages) { stage = 0; phase ^= 1u; stage_off = 0; }
    }
}

// Weights are read once per forward (350 MB per step > L2), so the first touch of every B tile would pay the HBM round
// trip inside a latency-bound main loop.  Each launch therefore pulls the weight matrices of the NEXT GEMM step of the
// plan into L2 while it computes: every CTA prefetches its 1/ctas slice of each matrix (one bulk-prefetch instruction
// per matrix, issued by one otherwise idle epilogue lane before the dependency wait - weights never change).
__device__ __forceinline__ void prefetch_next_weights(const GemmParams* __restrict__ next, int next_groups, int cta, int nctas) {
    for (int g = 0; g < next_groups; ++g) {
        const size_t bytes = (size_t)next[g].N * (size_t)next[g].b_ld * 2;
        size_t chunk = ((bytes + nctas - 1) / nctas + 127) & ~(size_t)127;
        const size_t off = (size_t)cta * chunk;
        if (off >= bytes) continue;
        if (off + chunk > bytes) chunk = (bytes - off) & ~(size_t)15;
        if (chunk) l2_prefetch_bulk(reinterpret_cast<const char*>(next[g].b_ptr) + off, (uint32_t)chunk);
    }
}

template <int ACT, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 2)
gemm_tc_kernel(const GemmParams* __restrict__ params, int stages, int kgroup, const GemmParams* __restrict__ next, int next_groups,
               int two_producers) {
    pdl_launch_dependents();
    if (next != nullptr && threadIdx.x == 64)
        prefetch_next_weights(next, next_groups, (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x, gridDim.x * gridDim.y * gridDim.z);
    const GemmParams& p = params[blockIdx.z];
    const int m_tile = blockIdx.x;
    const int n0 = blockIdx.y * p.block_n;
    if (m_tile * kBlockM >= p.M || n0 >= p.N) return;   // grouped launches: grid is sized for the largest member

    // no static shared memory in this kernel, so the declared alignment puts the dynamic window on a 1024-byte boundary
    // (SWIZZLE_128B atoms); checked rather than padded: the 1 KB matters for the two-CTA-per-SM configurations
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((smem_u32(smem) & 1023u) != 0u) { if (threadIdx.x == 0) printf("tmae: dynamic shared memory not 1024-byte aligned\n"); __trap(); }
    const int block_n = p.block_n;
    const bool reuse = p.in_mode == IN_CONV && p.conv_reuse != 0;
    const uint32_t reuse_a_bytes = reuse ? (uint32_t)(p.a_halo_rows * kBlockK * 2) : 0u;
    const int stage_bytes = reuse ? (int)reuse_a_bytes + 3 * block_n * kBlockK * 2 : kgroup * (kAStageBytes + block_n * kBlockK * 2);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)stages * stage_bytes);
    uint64_t* empty_bar = full_bar + stages;
    uint64_t* accum_bar = empty_bar + stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    long long* ticks = p.dbg_ticks ? p.dbg_ticks + ((size_t)(blockIdx.y * gridDim.x + blockIdx.x)) * 16 : nullptr;
    if (ticks && threadIdx.x == 0) ticks[0] = globaltimer_ns();

    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)block_n) tmem_cols <<= 1;

    int kb_per_tap = 0;
    for (int sg = 0; sg < p.num_segs; ++sg) kb_per_tap += p.seg_kblocks[sg];
    const int total_kb = kb_per_tap * p.num_taps;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        mbar_init(accum_bar, 1);
        fence_barrier_init();
        for (int sg = 0; sg < p.num_segs; ++sg) tma_prefetch_desc(&p.a_map[sg]);
        tma_prefetch_desc(&p.b_map);
    }
    if (warp == 1) {
        tmem_alloc(tmem_slot, tmem_cols);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (ticks && threadIdx.x == 0) ticks[1] = globaltimer_ns();
    pdl_wait();                 // everything above overlapped the previous kernel's tail; its outputs are visible from here

    // Producer and MMA loops are WARP-UNIFORM (all 32 lanes run the loop on identical values, only the TMA / MMA /
    // commit instructions are elect-predicated), so the compiler keeps addresses and descriptors in uniform registers
    // instead of moving them from a divergent lane for every instruction.
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t full_a = smem_u32(full_bar), empty_a = smem_u32(empty_bar);
    const int num_prod = (two_producers && total_kb > (reuse ? 3 : kgroup)) ? 2 : 1;
    if (warp == 0) {
        // ===== TMA producer =====
        int stage = 0;
        uint32_t phase = 0, stage_off = 0;
        produce_tile(p, m_tile, n0, total_kb, stages, kgroup, stage_bytes, smem_base, full_a, empty_a, stage, phase, stage_off, ticks,
                     0, num_prod);
    } else if (warp == 1) {
        // ===== MMA issuer =====
        int stage = 0;
        uint32_t phase = 0, stage_off = 0;
        mma_tile(block_n, total_kb, stages, kgroup, stage_bytes, smem_base, full_a, empty_a, tmem_base, smem_u32(accum_bar),
                 stage, phase, stage_off, ticks, 3, 4, reuse_a_bytes, (uint32_t)(p.box_n * p.s * kBlockK * 2));
    } else {
        // ===== epilogue (warps 2..9; TMEM lane quarter = warp % 4, two warps per quarter alternate 32-column chunks) =====
        // Phase 1 (thread = accumulator row): TMEM -> registers -> smem staging tile (raw fp32 accumulators).
        // Phase 2 (8 lanes = 32 consecutive channels of one row, 4 rows per instruction): + bias, activation,
        // residual add, coalesced 64 / 128-byte row segments to global memory.  The staging tiles reuse the (now
        // idle) pipeline buffers: accum_bar completes only after every MMA has finished reading them.
        // The staging tiles reuse the (now idle) pipeline buffers: accum_bar completes only after every MMA has
        // finished reading them.
        if (warp == 2 && num_prod == 2) {             // second producer: an epilogue warp, idle until the accumulator is done
            int stage = 0;
            uint32_t phase = 0, stage_off = 0;
            produce_tile(p, m_tile, n0, total_kb, stages, kgroup, stage_bytes, smem_base, full_a, empty_a, stage, phase, stage_off,
                         nullptr, 1, 2);
        }
        const EpiCtx e = load_epi(p);
        epilogue_tile<ACT, EPI>(e, m_tile, n0, block_n, tmem_base, smem_base, warp, lane, accum_bar, 0u, ticks);
        if (ticks && warp == 2 && lane == 0) ticks[6] = globaltimer_ns();
    }
    tc_fence_before();
    __syncthreads();
    if (ticks && threadIdx.x == 0) ticks[7] = globaltimer_ns();
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// ---------------------------------------------------------------------------------------------------------
// Persistent variant for launches with several tiles per SM (encoder QKV / fc1): one CTA per SM walks a static
// round-robin tile list; the smem pipeline runs straight across tile boundaries and the accumulator is double
// buffered in TMEM (2 x 256 columns), so the epilogue of tile i overlaps the main loop of tile i+1.
//   barriers: full/empty[stages] (TMA <-> MMA), tfull/tempty[2] (MMA <-> epilogue)
// ---------------------------------------------------------------------------------------------------------
constexpr int kPersistEpiWarps = 16;                       // 4 warps per TMEM lane quarter: the GELU epilogue of fc1 is issue bound
constexpr int kPersistThreads = 64 + 32 * kPersistEpiWarps;
constexpr int kEpiStageBytes = kPersistEpiWarps * 32 * kEpiPitch * 4;   // dedicated staging tiles (the pipeline never idles here)

template <int ACT, int EPI>
__global__ void __launch_bounds__(kPersistThreads, 1)
gemm_tc_persistent_kernel(const GemmParams* __restrict__ params, int stages, int m_tiles, int n_tiles, const GemmParams* __restrict__ next, int next_groups) {
    pdl_launch_dependents();
    if (next != nullptr && threadIdx.x == 64) prefetch_next_weights(next, next_groups, blockIdx.x, gridDim.x);
    const GemmParams& p = params[0];
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int block_n = p.block_n;
    const int stage_bytes = kAStageBytes + block_n * kBlockK * 2;
    uint8_t* pipe = smem + kEpiStageBytes;                    // a multiple of 1024 B: the stages keep their swizzle alignment
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(pipe + (size_t)stages * stage_bytes);
    uint64_t* empty_bar = full_bar + stages;
    uint64_t* tfull_bar = empty_bar + stages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    int kb_per_tap = 0;
    for (int sg = 0; sg < p.num_segs; ++sg) kb_per_tap += p.seg_kblocks[sg];
    const int total_kb = kb_per_tap * p.num_taps;
    const int total_tiles = m_tiles * n_tiles;
    long long* ticks = p.dbg_ticks ? p.dbg_ticks + (size_t)blockIdx.x * 16 : nullptr;
    if (ticks && threadIdx.x == 0) ticks[0] = globaltimer_ns();

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], kPersistEpiWarps); }
        fence_barrier_init();
        for (int sg = 0; sg < p.num_segs; ++sg) tma_prefetch_desc(&p.a_map[sg]);
        tma_prefetch_desc(&p.b_map);
    }
    if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();
    const uint32_t pipe_base = smem_u32(pipe);
    const uint32_t full_a = smem_u32(full_bar), empty_a = smem_u32(empty_bar);

    if (warp == 0) {
        // ===== TMA producer (warp-uniform) =====
        int stage = 0;
        uint32_t phase = 0, stage_off = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x)
            produce_tile(p, t / n_tiles, (t % n_tiles) * block_n, total_kb, stages, 1, stage_bytes, pipe_base, full_a, empty_a,
                         stage, phase, stage_off, nullptr);
    } else if (warp == 1) {
        // ===== MMA issuer (warp-uniform) =====
        int stage = 0, it = 0;
        uint32_t phase = 0, stage_off = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
            mbar_wait(&tempty_bar[buf], acc_phase ^ 1u);           // epilogue has drained this accumulator buffer
            tc_fence_after();
            mma_tile(block_n, total_kb, stages, 1, stage_bytes, pipe_base, full_a, empty_a, tmem_base + (uint32_t)buf * 256u,
                     smem_u32(&tfull_bar[buf]), stage, phase, stage_off, it < 3 ? ticks : nullptr, 1 + 4 * it, 2 + 4 * it);
        }
    } else {
        // ===== epilogue warps =====
        const EpiCtx e = load_epi(p);
        const uint32_t stage_base = smem_u32(smem);
        int it = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
            const int m_tile = t / n_tiles, n0 = (t % n_tiles) * block_n;
            long long tk[16];
            epilogue_tile<ACT, EPI>(e, m_tile, n0, block_n, tmem_base + (uint32_t)buf * 256u, stage_base, warp, lane,
                                    &tfull_bar[buf], acc_phase, (ticks && warp == 2 && it < 3) ? tk : nullptr, kPersistEpiWarps / 4);
            if (ticks && warp == 2 && lane == 0 && it < 3) { ticks[3 + 4 * it] = tk[5]; ticks[4 + 4 * it] = globaltimer_ns(); }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[buf]);           // one arrival per epilogue warp frees the buffer
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05.mma.cta_group::2) for the linear layers with many rows (encoder QKV / proj / fc1 / fc2):
// a cluster of two CTAs (the two SMs of a TPC) computes ONE 256 x block_n tile.  CTA r stages rows [128 r, 128 r + 128) of
// the A tile and rows [r block_n / 2, (r + 1) block_n / 2) of the weight tile; the leader (cluster rank 0) issues the MMAs,
// which read both CTAs' shared memory and write each CTA's half of the accumulator into that CTA's tensor memory.
// Per SM and k-block that is 16 KB + 64 block_n bytes through the shared-memory port instead of 16 KB + 128 block_n for
// the same flops - the 1-CTA tile is shared-memory-bandwidth bound (DESIGN.md 3).
//   full[s]   in the LEADER: armed by the leader's producer with the bytes of both CTAs, completed by both CTAs' TMA loads
//   empty[s]  in each CTA: tcgen05.commit multicast from the leader's MMA warp frees the stage in both
//   accum     in each CTA: multicast commit after the last MMA; each CTA's epilogue drains its own 128 TMEM lanes
// ---------------------------------------------------------------------------------------------------------
template <int ACT, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 2)
gemm_tc_pair_kernel(const GemmParams* __restrict__ params, int stages, const GemmParams* __restrict__ next, int next_groups) {
    pdl_launch_dependents();
    if (next != nullptr && threadIdx.x == 64)
        prefetch_next_weights(next, next_groups, (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x, gridDim.x * gridDim.y * gridDim.z);
    const GemmParams& p = params[blockIdx.z];
    const uint32_t rank = cluster_ctarank();             // cluster = 2 consecutive CTAs along x
    const int m_tile = blockIdx.x;                       // this CTA's 128 rows (conv: its box of images / rows): pair blockIdx.x / 2, half `rank`
    const int n0 = blockIdx.y * p.block_n;
    if ((m_tile >> 1) * 2 * kBlockM >= p.M || n0 >= p.N) return;      // uniform over the pair (grouped launches: smaller members)

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((smem_u32(smem) & 1023u) != 0u) { if (threadIdx.x == 0) printf("tmae: dynamic shared memory not 1024-byte aligned\n"); __trap(); }
    const int block_n = p.block_n;
    const int half_n = block_n >> 1;
    const bool reuse = p.in_mode == IN_CONV && p.conv_reuse != 0;
    const uint32_t reuse_a_bytes = reuse ? (uint32_t)(p.a_halo_rows * kBlockK * 2) : 0u;
    const int stage_bytes = reuse ? (int)reuse_a_bytes + 3 * half_n * kBlockK * 2 : kAStageBytes + half_n * kBlockK * 2;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)stages * stage_bytes);
    uint64_t* empty_bar = full_bar + stages;
    uint64_t* accum_bar = empty_bar + stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)block_n) tmem_cols <<= 1;
    int total_kb = 0;
    for (int sg = 0; sg < p.num_segs; ++sg) total_kb += p.seg_kblocks[sg];
    total_kb *= p.num_taps;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        mbar_init(accum_bar, 1);
        fence_barrier_init();
        for (int sg = 0; sg < p.num_segs; ++sg) tma_prefetch_desc(&p.a_map[sg]);
        tma_prefetch_desc(&p.b_map_pair);
    }
    if (warp == 1) { tmem_alloc_pair(tmem_slot, tmem_cols); tmem_relinquish_pair(); }
    tc_fence_before();
    cluster_sync_all();                                   // both CTAs' barriers exist before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();

    const uint32_t smem_base = smem_u32(smem);
    const uint32_t full_a = smem_u32(full_bar), empty_a = smem_u32(empty_bar);
    if (warp == 0) {
        // ===== TMA producer (both CTAs) =====
        int stage = 0;
        uint32_t phase = 0, stage_off = 0;
        produce_tile(p, m_tile, n0, total_kb, stages, 1, stage_bytes, smem_base, full_a, empty_a, stage, phase, stage_off, nullptr,
                     0, 1, 1, rank, mapa_shared(full_a, 0));
    } else if (warp == 1) {
        if (rank == 0) {
            // ===== MMA issuer (leader only) =====
            int stage = 0;
            uint32_t phase = 0, stage_off = 0;
            mma_tile(block_n, total_kb, stages, 1, stage_bytes, smem_base, full_a, empty_a, tmem_base, smem_u32(accum_bar),
                     stage, phase, stage_off, nullptr, -1, -1, reuse_a_bytes, (uint32_t)(p.box_n * p.s * kBlockK * 2), 1);
        }
    } else {
        // ===== epilogue (both CTAs, own TMEM lanes = own 128 rows); staging reuses the idle pipeline buffers =====
        const EpiCtx e = load_epi(p);
        epilogue_tile<ACT, EPI>(e, m_tile, n0, block_n, tmem_base, smem_base, warp, lane, accum_bar, 0u, nullptr);
    }
    tc_fence_before();
    cluster_sync_all();                                   // neither CTA leaves while the other may still signal its barriers
    if (warp == 1) tmem_dealloc_pair(tmem_base, tmem_cols);
}

// ---------------------------------------------------------------------------------------------------------
// Persistent CTA-pair variant (encoder QKV / fc1 with one batch in flight): 74 clusters of two CTAs walk a static round-robin
// list of 256 x block_n tiles.  It combines the two mechanisms above: the pair halves the weight traffic per SM, and the
// accumulator is double buffered in tensor memory (2 x 256 columns in EACH CTA) so the 16 epilogue warps of a CTA drain tile
// i while the pair's main loop runs tile i + 1 - in the one-tile-per-CTA pair kernel the two phases alternate (main loop
// 7 us, store phase 3-7 us per tile) and the second wave of a 1.3-wave grid leaves most SMs idle.
//   full[s]    in the LEADER, completed by both CTAs' TMA loads          empty[s]  in each CTA (multicast commit)
//   tfull[b]   in each CTA (multicast commit after the tile's last MMA)  tempty[b] in the LEADER: 2 x 16 arrivals, one per
//              epilogue warp of BOTH CTAs (the follower's arrive through the cluster address)
// ---------------------------------------------------------------------------------------------------------
template <int ACT, int EPI>
__global__ void __launch_bounds__(kPersistThreads, 1)
gemm_tc_pair_persistent_kernel(const GemmParams* __restrict__ params, int stages, int m_pairs, int n_tiles,
                               const GemmParams* __restrict__ next, int next_groups) {
    pdl_launch_dependents();
    if (next != nullptr && threadIdx.x == 64) prefetch_next_weights(next, next_groups, blockIdx.x, gridDim.x);
    const GemmParams& p = params[0];
    const uint32_t rank = cluster_ctarank();
    const int pair_id = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int block_n = p.block_n;
    const int half_n = block_n >> 1;
    const int stage_bytes = kAStageBytes + half_n * kBlockK * 2;
    uint8_t* pipe = smem + kEpiStageBytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(pipe + (size_t)stages * stage_bytes);
    uint64_t* empty_bar = full_bar + stages;
    uint64_t* tfull_bar = empty_bar + stages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    int total_kb = 0;
    for (int sg = 0; sg < p.num_segs; ++sg) total_kb += p.seg_kblocks[sg];
    total_kb *= p.num_taps;
    const int total_tiles = m_pairs * n_tiles;
    long long* ticks = p.dbg_ticks ? p.dbg_ticks + (size_t)blockIdx.x * 16 : nullptr;     // bring-up: phase stamps of the first 3 tiles
    if (ticks && threadIdx.x == 0) ticks[0] = globaltimer_ns();

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * kPersistEpiWarps); }
        fence_barrier_init();
        for (int sg = 0; sg < p.num_segs; ++sg) tma_prefetch_desc(&p.a_map[sg]);
        tma_prefetch_desc(&p.b_map_pair);
    }
    if (warp == 1) { tmem_alloc_pair(tmem_slot, 512); tmem_relinquish_pair(); }
    tc_fence_before();
    cluster_sync_all();                                   // both CTAs' barriers exist before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();
    const uint32_t pipe_base = smem_u32(pipe);
    const uint32_t full_a = smem_u32(full_bar), empty_a = smem_u32(empty_bar);

    if (warp == 0) {
        // ===== TMA producer (both CTAs): own 128 rows of A, own half of the weight tile =====
        int stage = 0;
        uint32_t phase = 0, stage_off = 0;
        const uint32_t full_leader = mapa_shared(full_a, 0);
        for (int t = pair_id; t < total_tiles; t += num_pairs)
            produce_tile(p, 2 * (t / n_tiles) + (int)rank, (t % n_tiles) * block_n, total_kb, stages, 1, stage_bytes, pipe_base, full_a, empty_a,
                         stage, phase, stage_off, nullptr, 0, 1, 1, rank, full_leader);
    } else if (warp == 1) {
        if (rank == 0) {
            // ===== MMA issuer (leader only) =====
            int stage = 0, it = 0;
            uint32_t phase = 0, stage_off = 0;
            for (int t = pair_id; t < total_tiles; t += num_pairs, ++it) {
                const int buf = it & 1;
                const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
                mbar_wait_cluster(&tempty_bar[buf], acc_phase ^ 1u);      // both CTAs' epilogues have drained this buffer
                tc_fence_after();
                mma_tile(block_n, total_kb, stages, 1, stage_bytes, pipe_base, full_a, empty_a, tmem_base + (uint32_t)buf * 256u,
                         smem_u32(&tfull_bar[buf]), stage, phase, stage_off, it < 3 ? ticks : nullptr, 1 + 4 * it, 2 + 4 * it, 0u, 0u, 1);
            }
        }
    } else {
        // ===== epilogue warps (both CTAs, own TMEM lanes = own 128 rows) =====
        const EpiCtx e = load_epi(p);
        const uint32_t stage_base = smem_u32(smem);
        const uint32_t tempty_leader = mapa_shared(smem_u32(tempty_bar), 0);
        int it = 0;
        for (int t = pair_id; t < total_tiles; t += num_pairs, ++it) {
            const int buf = it & 1;
            const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
            long long tk[16];
            epilogue_tile<ACT, EPI>(e, 2 * (t / n_tiles) + (int)rank, (t % n_tiles) * block_n, block_n, tmem_base + (uint32_t)buf * 256u,
                                    stage_base, warp, lane, &tfull_bar[buf], acc_phase, (ticks && warp == 2 && it < 3) ? tk : nullptr,
                                    kPersistEpiWarps / 4);
            if (ticks && warp == 2 && lane == 0 && it < 3) { ticks[3 + 4 * it] = tk[5]; ticks[4 + 4 * it] = globaltimer_ns(); }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty_leader + 8u * (uint32_t)buf);
        }
    }
    tc_fence_before();
    cluster_sync_all();                                   // neither CTA leaves while the other may still signal its barriers
    if (ticks && threadIdx.x == 0) ticks[13] = globaltimer_ns();
    if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------------
// CUDA-core checker: same parameter block, same epilogue, plain loads.  Bring-up / tests only.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
gemm_simt_kernel(const GemmParams* __restrict__ params) {
    pdl_wait();
    const GemmParams& p = params[blockIdx.z];
    const int m = blockIdx.x;
    if (m >= p.M) return;
    const EpiCtx e = load_epi(p);
    const RowCtx r = decode_row(e, m / kBlockM, m % kBlockM);
    if (!r.valid) return;
    const bool conv = p.in_mode == IN_CONV;
    for (int col = threadIdx.x * 8; col < p.N; col += blockDim.x * 8) {
        float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int tap = 0; tap < p.num_taps; ++tap) {
            long long row = r.lin;
            if (conv) {                                          // zero padding: taps outside the image contribute nothing
                const int yy = r.y + tap / 3 - 1, xx = r.x + tap % 3 - 1;
                row = (yy >= 0 && yy < p.s && xx >= 0 && xx < p.s) ? (long long)r.n * p.K + yy * p.s + xx : -1;
            }
            for (int sg = 0; sg < p.num_segs; ++sg) {
                const int kbase = (tap * p.b_kb_per_tap + p.seg_b_kb0[sg]) * kBlockK;
                if (row >= 0 && row < p.a_rows[sg]) {
                    const __nv_bfloat16* a = p.a_ptr[sg] + row * p.a_ld[sg];
                    for (int c = 0; c < p.a_cols[sg]; ++c) {
                        const float av = __bfloat162float(a[c]);
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            v[i] = fmaf(av, __bfloat162float(p.b_ptr[(long long)(col + i) * p.b_ld + kbase + c]), v[i]);
                    }
                }
            }
        }
        epilogue8(e, r, col, v);
    }
}

// ---------------------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------------------
// conv_reuse launches: a stage is one haloed A box + three B atoms (`stage_bytes`); returns 0 if fewer than 2 fit
int gemm_reuse_stages(int stage_bytes, int total_ctas, bool share_sm, int* smem_bytes) {
    const int overhead = 256;
    const bool whole_sm = total_ctas <= 148 && !share_sm;
    const int budget = (whole_sm ? 226 : 113) * 1024 - overhead;
    int stages = budget / stage_bytes;
    if (stages > 4) stages = 4;                    // 12 k-blocks in flight
    if (stages < 2) return 0;
    *smem_bytes = overhead + stages * stage_bytes;
    return stages;
}

int gemm_pick_stages(int block_n, int total_ctas, bool share_sm, int* smem_bytes, int* kgroup) {
    // Small tiles are bound by (a) the TMA round trip: bytes in flight per SM is what matters, and (b) the ~300-cycle
    // producer <-> MMA handshake per pipeline stage: see produce_tile.  A single wave (<= 148 CTAs) gets the whole
    // shared memory of its SM; larger grids run two CTAs per SM so that one CTA's epilogue overlaps the other's loop.
    // share_sm: several handles / streams are in flight on this GPU, so even a single-wave launch keeps to half the
    // shared memory and lets a CTA of another stream's kernel co-reside (measured +9 % throughput at 3 streams).
    static const int force_g = getenv("TMAE_KGROUP") ? atoi(getenv("TMAE_KGROUP")) : 0;
    const int atom = kAStageBytes + block_n * kBlockK * 2;
    const int overhead = 256;                       // barriers + TMEM slot (the pipeline itself starts at offset 0)
    const bool whole_sm = total_ctas <= 148 && !share_sm;
    const int budget = (whole_sm ? 226 : 113) * 1024 - overhead;
    const int max_kb_in_flight = whole_sm ? 10 : 6;
    // two k-blocks per handshake once their 8 MMAs (128 x block_n / 32 cycles) no longer cover it, if >= 3 (whole SM) /
    // >= 2 (half SM, the co-resident CTA fills the bubbles) such stages still fit
    int g = 1;
    if (block_n <= 128 && budget / (2 * atom) >= (whole_sm ? 3 : 2)) g = 2;
    if (force_g == 1 || force_g == 2 || force_g == 4) { g = force_g; while (g > 1 && budget / (g * atom) < 2) g >>= 1; }
    int stages = budget / (g * atom);
    if (stages * g > max_kb_in_flight) stages = max_kb_in_flight / g;
    if (stages < 2) stages = 2;
    *kgroup = g;
    *smem_bytes = overhead + stages * g * atom;
    return stages;
}

template <int ACT, int EPI>
static cudaError_t configure_one() {
    prefer_max_smem_carveout(gemm_tc_kernel<ACT, EPI>);
    return cudaFuncSetAttribute(gemm_tc_kernel<ACT, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

cudaError_t gemm_tc_configure() {
    cudaError_t e;
    if ((e = configure_one<ACT_NONE, EPI_GENERIC>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_GELU, EPI_GENERIC>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_HALF_TANH, EPI_GENERIC>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_NONE, EPI_BF16_SAME>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_GELU, EPI_BF16_SAME>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_NONE, EPI_F32_SAME_RESID>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_NONE, EPI_GAUSS>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_NONE, EPI_GAUSS_IDX>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_NONE, EPI_BF16_TMA>()) != cudaSuccess) return e;
    if ((e = configure_one<ACT_GELU, EPI_BF16_TMA>()) != cudaSuccess) return e;
    {
        auto cfgp = [](auto kern) {
            prefer_max_smem_carveout(kern);
            return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        };
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_NONE, EPI_BF16_TMA>)) != cudaSuccess) return e;
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_GELU, EPI_BF16_TMA>)) != cudaSuccess) return e;
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_NONE, EPI_BF16_SAME>)) != cudaSuccess) return e;
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_GELU, EPI_BF16_SAME>)) != cudaSuccess) return e;
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_NONE, EPI_F32_SAME_RESID>)) != cudaSuccess) return e;
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_NONE, EPI_GENERIC>)) != cudaSuccess) return e;
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_GELU, EPI_GENERIC>)) != cudaSuccess) return e;
        if ((e = cfgp(gemm_tc_pair_kernel<ACT_HALF_TANH, EPI_GENERIC>)) != cudaSuccess) return e;
    }
    {
        auto cfgpp = [](auto kernel) {
            prefer_max_smem_carveout(kernel);
            return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        };
        if ((e = cfgpp(gemm_tc_pair_persistent_kernel<ACT_NONE, EPI_BF16_TMA>)) != cudaSuccess) return e;
        if ((e = cfgpp(gemm_tc_pair_persistent_kernel<ACT_GELU, EPI_BF16_TMA>)) != cudaSuccess) return e;
        if ((e = cfgpp(gemm_tc_pair_persistent_kernel<ACT_NONE, EPI_BF16_SAME>)) != cudaSuccess) return e;
        if ((e = cfgpp(gemm_tc_pair_persistent_kernel<ACT_GELU, EPI_BF16_SAME>)) != cudaSuccess) return e;
    }
    prefer_max_smem_carveout(gemm_tc_persistent_kernel<ACT_NONE, EPI_BF16_TMA>);
    prefer_max_smem_carveout(gemm_tc_persistent_kernel<ACT_GELU, EPI_BF16_TMA>);
    if ((e = cudaFuncSetAttribute(gemm_tc_persistent_kernel<ACT_NONE, EPI_BF16_TMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(gemm_tc_persistent_kernel<ACT_GELU, EPI_BF16_TMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    prefer_max_smem_carveout(gemm_tc_persistent_kernel<ACT_NONE, EPI_BF16_SAME>);
    prefer_max_smem_carveout(gemm_tc_persistent_kernel<ACT_GELU, EPI_BF16_SAME>);
    if ((e = cudaFuncSetAttribute(gemm_tc_persistent_kernel<ACT_NONE, EPI_BF16_SAME>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(gemm_tc_persistent_kernel<ACT_GELU, EPI_BF16_SAME>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

// Persistent launch qualifies: one group, bf16 same-row output, more tiles than 2 per SM.
// Not used when several streams share the GPU: a persistent launch owns every SM (one CTA, all of its shared memory),
// which removes the cross-stream overlap that mode relies on (measured: 26.5k vs 25.9k images/s at 3 streams).
bool gemm_use_persistent(int groups, int epi, int act, int tiles, bool share_sm) {
    static const bool off = getenv("TMAE_NO_PERSISTENT") != nullptr;
    return !off && !share_sm && groups == 1 && (epi == EPI_BF16_SAME || epi == EPI_BF16_TMA) && (act == ACT_NONE || act == ACT_GELU) && tiles > 2 * 148;
}

// Store-phase specialisation a parameter block qualifies for (every member of a grouped launch must agree).
int gemm_epi_kind(const GemmParams& p) {
    if (p.gc_on) return p.gc_on == 2 ? EPI_GAUSS_IDX : EPI_GAUSS;
    const bool one_out = p.out[1].dtype == OUT_NONE && p.out[0].map == MAP_SAME;
    static const bool no_tma_store = getenv("TMAE_NO_TMA_STORE") != nullptr;
    if (one_out && p.out[0].dtype == OUT_BF16 && p.resid == nullptr && p.act != ACT_HALF_TANH)
        return (p.tma_store_ok && (p.block_n & 31) == 0 && !no_tma_store) ? EPI_BF16_TMA : EPI_BF16_SAME;
    if (one_out && p.in_mode != IN_CONV && p.out[0].dtype == OUT_F32 && p.resid != nullptr && p.resid_map == MAP_SAME && p.act == ACT_NONE)
        return EPI_F32_SAME_RESID;
    return EPI_GENERIC;
}

// CTA-pair policy.  Linear layers: one bf16 / fp32+residual same-row output and >= 8 row tiles (the encoder GEMMs).  3x3 conv
// layers: >= 8 row tiles and a weight tile of >= 64 columns (below that the B tile is too small for halving it to matter and
// the launch is latency bound).  block_n % 16 == 0 always holds.  TMAE_NO_PAIR=1 / TMAE_NO_PAIR_CONV=1 switch them off (A/B).
bool gemm_use_pair(int groups, int epi, int act, int max_M, int block_n, bool pair_ok, bool conv) {
    static const bool off = getenv("TMAE_NO_PAIR") != nullptr;
    static const bool off_conv = getenv("TMAE_NO_PAIR_CONV") != nullptr;
    if (off || !pair_ok || max_M < 8 * kBlockM) return false;
    if (conv) return !off_conv && block_n >= 64;
    if (groups != 1) return false;
    if (epi == EPI_F32_SAME_RESID) return act == ACT_NONE;
    return (epi == EPI_BF16_SAME || epi == EPI_BF16_TMA) && (act == ACT_NONE || act == ACT_GELU);
}

// Persistent pairs: a linear layer that already qualifies for pairs, bf16 same-row output, one batch in flight (a persistent
// launch owns every SM) and more pair tiles than one round of the 74 clusters.  TMAE_NO_PAIR_PERSISTENT=1 = A/B switch.
bool gemm_use_pair_persistent(int groups, int epi, int act, int max_M, int max_N, int block_n, bool share_sm, bool conv) {
    static const bool off = getenv("TMAE_NO_PAIR_PERSISTENT") != nullptr;
    static const bool in_share = getenv("TMAE_PP_SHARE") != nullptr;          // experiment: also while several streams share the GPU
    if (off || (share_sm && !in_share) || conv || groups != 1) return false;
    if ((epi != EPI_BF16_SAME && epi != EPI_BF16_TMA) || (act != ACT_NONE && act != ACT_GELU)) return false;
    const int m_pairs = ((max_M + kBlockM - 1) / kBlockM + 1) / 2, n_tiles = (max_N + block_n - 1) / block_n;
    return m_pairs * n_tiles > 74;
}

template <int ACT, int EPI>
static cudaError_t launch_pair(dim3 grid, int smem, cudaStream_t stream, const GemmParams* d_params, int stages, const GemmParams* d_next,
                               int next_groups) {
    return launch_k_cluster(gemm_tc_pair_kernel<ACT, EPI>, grid, dim3(kGemmThreads), smem, stream, true, 2, d_params, stages, d_next, next_groups);
}

// params: device array of `groups` GemmParams; max_M / max_N / block_n describe the largest member.
cudaError_t gemm_launch(const GemmParams* d_params, int groups, int max_M, int max_N, int block_n, int act, int epi,
                        bool simt, bool share_sm, cudaStream_t stream, const GemmParams* d_next, int next_groups,
                        int conv_reuse_stage_bytes, int pair) {
    if (simt) {
        dim3 grid(max_M, 1, groups);
        gemm_simt_kernel<<<grid, 128, 0, stream>>>(d_params);
        return cudaGetLastError();
    }
    int smem = 0;
    dim3 grid((max_M + kBlockM - 1) / kBlockM, (max_N + block_n - 1) / block_n, groups);
    if (pair) {                                               // the plan's policy (gemm_use_pair) decided
        if ((block_n & 15) != 0) return cudaErrorInvalidConfiguration;
        dim3 pgrid((grid.x + 1) / 2 * 2, grid.y, groups);      // whole pairs along x
        if (pair == 2) {
            // persistent pairs (plan policy gemm_use_pair_persistent): one cluster per TPC, tiles round-robin
            if (groups != 1 || conv_reuse_stage_bytes != 0 || (epi != EPI_BF16_SAME && epi != EPI_BF16_TMA) || (act != ACT_NONE && act != ACT_GELU))
                return cudaErrorInvalidConfiguration;
            const int stage_bytes = kAStageBytes + (block_n / 2) * kBlockK * 2;
            const int overhead = 1024 + 256 + kEpiStageBytes;
            int pst = (226 * 1024 - overhead) / stage_bytes;
            if (pst > 8) pst = 8;
            if (pst < 2) return cudaErrorInvalidConfiguration;
            const int psmem = overhead + pst * stage_bytes;
            const int m_pairs = (int)pgrid.x / 2, tiles = m_pairs * (int)grid.y;
            const int pairs = tiles < 74 ? tiles : 74;
            const dim3 g2(2 * pairs), blk(kPersistThreads);
            if (epi == EPI_BF16_TMA && act == ACT_GELU) return launch_k_cluster(gemm_tc_pair_persistent_kernel<ACT_GELU, EPI_BF16_TMA>, g2, blk, psmem, stream, true, 2, d_params, pst, m_pairs, (int)grid.y, d_next, next_groups);
            if (epi == EPI_BF16_TMA) return launch_k_cluster(gemm_tc_pair_persistent_kernel<ACT_NONE, EPI_BF16_TMA>, g2, blk, psmem, stream, true, 2, d_params, pst, m_pairs, (int)grid.y, d_next, next_groups);
            if (act == ACT_GELU) return launch_k_cluster(gemm_tc_pair_persistent_kernel<ACT_GELU, EPI_BF16_SAME>, g2, blk, psmem, stream, true, 2, d_params, pst, m_pairs, (int)grid.y, d_next, next_groups);
            return launch_k_cluster(gemm_tc_pair_persistent_kernel<ACT_NONE, EPI_BF16_SAME>, g2, blk, psmem, stream, true, 2, d_params, pst, m_pairs, (int)grid.y, d_next, next_groups);
        }
        // conv_reuse_stage_bytes is the PAIR stage here (haloed A box + three half B atoms), computed by the plan
        const int stage_bytes = conv_reuse_stage_bytes > 0 ? conv_reuse_stage_bytes : kAStageBytes + (block_n / 2) * kBlockK * 2;
        const int overhead = 256;
        const bool whole_sm = (int)(pgrid.x * pgrid.y * pgrid.z) <= 148 && !share_sm;
        const int budget = (whole_sm ? 226 : 113) * 1024 - overhead;
        int pst = budget / stage_bytes;
        if (pst > (conv_reuse_stage_bytes > 0 ? 4 : 8)) pst = conv_reuse_stage_bytes > 0 ? 4 : 8;
        if (pst < 2) return cudaErrorInvalidConfiguration;
        const int psmem = overhead + pst * stage_bytes;
        if (epi == EPI_BF16_TMA) return act == ACT_GELU ? launch_pair<ACT_GELU, EPI_BF16_TMA>(pgrid, psmem, stream, d_params, pst, d_next, next_groups)
                                                        : launch_pair<ACT_NONE, EPI_BF16_TMA>(pgrid, psmem, stream, d_params, pst, d_next, next_groups);
        if (epi == EPI_BF16_SAME) return act == ACT_GELU ? launch_pair<ACT_GELU, EPI_BF16_SAME>(pgrid, psmem, stream, d_params, pst, d_next, next_groups)
                                                         : launch_pair<ACT_NONE, EPI_BF16_SAME>(pgrid, psmem, stream, d_params, pst, d_next, next_groups);
        if (epi == EPI_F32_SAME_RESID) return launch_pair<ACT_NONE, EPI_F32_SAME_RESID>(pgrid, psmem, stream, d_params, pst, d_next, next_groups);
        if (act == ACT_GELU) return launch_pair<ACT_GELU, EPI_GENERIC>(pgrid, psmem, stream, d_params, pst, d_next, next_groups);
        if (act == ACT_HALF_TANH) return launch_pair<ACT_HALF_TANH, EPI_GENERIC>(pgrid, psmem, stream, d_params, pst, d_next, next_groups);
        return launch_pair<ACT_NONE, EPI_GENERIC>(pgrid, psmem, stream, d_params, pst, d_next, next_groups);
    }
    if (conv_reuse_stage_bytes == 0 && gemm_use_persistent(groups, epi, act, (int)(grid.x * grid.y), share_sm)) {
        const int stage_bytes = kAStageBytes + block_n * kBlockK * 2;
        const int overhead = 1024 + 256 + kEpiStageBytes;
        int pst = (226 * 1024 - overhead) / stage_bytes;
        if (pst > 8) pst = 8;
        const int psmem = overhead + pst * stage_bytes;
        const int tiles = (int)(grid.x * grid.y);
        const int ctas = tiles < 148 ? tiles : 148;
        if (epi == EPI_BF16_TMA && act == ACT_GELU) return launch_k(gemm_tc_persistent_kernel<ACT_GELU, EPI_BF16_TMA>, dim3(ctas), dim3(kPersistThreads), psmem, stream, true, d_params, pst, (int)grid.x, (int)grid.y, d_next, next_groups);
        if (epi == EPI_BF16_TMA) return launch_k(gemm_tc_persistent_kernel<ACT_NONE, EPI_BF16_TMA>, dim3(ctas), dim3(kPersistThreads), psmem, stream, true, d_params, pst, (int)grid.x, (int)grid.y, d_next, next_groups);
        if (act == ACT_GELU) return launch_k(gemm_tc_persistent_kernel<ACT_GELU, EPI_BF16_SAME>, dim3(ctas), dim3(kPersistThreads), psmem, stream, true, d_params, pst, (int)grid.x, (int)grid.y, d_next, next_groups);
        return launch_k(gemm_tc_persistent_kernel<ACT_NONE, EPI_BF16_SAME>, dim3(ctas), dim3(kPersistThreads), psmem, stream, true, d_params, pst, (int)grid.x, (int)grid.y, d_next, next_groups);
    }
    static const int two_prod_env = getenv("TMAE_TWO_PRODUCERS") ? atoi(getenv("TMAE_TWO_PRODUCERS")) : -1;
    int kgroup = 1;
    int stages;
    if (conv_reuse_stage_bytes > 0) {
        stages = gemm_reuse_stages(conv_reuse_stage_bytes, (int)(grid.x * grid.y * grid.z), share_sm, &smem);
        if (stages == 0) return cudaErrorInvalidConfiguration;      // the plan only marks launches whose stages fit
    } else {
        stages = gemm_pick_stages(block_n, (int)(grid.x * grid.y * grid.z), share_sm, &smem, &kgroup);
    }
    // Second producer warp (TMAE_TWO_PRODUCERS=1): in isolation it shortens producer-bound main loops (64-wide GEMM
    // tiles -20 %, fc2 -8 %), but since the conv layers moved to one haloed A box per three taps the whole forward is
    // 4 % FASTER without it (25.6k vs 24.4k images/s, one batch in flight; equal with four) - off by default.
    const int two_prod = two_prod_env >= 0 ? two_prod_env : 0;
    // every member of a grouped launch shares the activation and the store-phase specialisation
    if (epi == EPI_GAUSS) return launch_k(gemm_tc_kernel<ACT_NONE, EPI_GAUSS>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    if (epi == EPI_GAUSS_IDX) return launch_k(gemm_tc_kernel<ACT_NONE, EPI_GAUSS_IDX>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    if (epi == EPI_BF16_TMA && act == ACT_GELU) return launch_k(gemm_tc_kernel<ACT_GELU, EPI_BF16_TMA>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    else if (epi == EPI_BF16_TMA && act == ACT_NONE) return launch_k(gemm_tc_kernel<ACT_NONE, EPI_BF16_TMA>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    else if (epi == EPI_BF16_SAME && act == ACT_GELU) return launch_k(gemm_tc_kernel<ACT_GELU, EPI_BF16_SAME>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    else if (epi == EPI_BF16_SAME && act == ACT_NONE) return launch_k(gemm_tc_kernel<ACT_NONE, EPI_BF16_SAME>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    else if (epi == EPI_F32_SAME_RESID && act == ACT_NONE) return launch_k(gemm_tc_kernel<ACT_NONE, EPI_F32_SAME_RESID>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    else if (act == ACT_GELU) return launch_k(gemm_tc_kernel<ACT_GELU, EPI_GENERIC>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    else if (act == ACT_HALF_TANH) return launch_k(gemm_tc_kernel<ACT_HALF_TANH, EPI_GENERIC>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    else return launch_k(gemm_tc_kernel<ACT_NONE, EPI_GENERIC>, grid, dim3(kGemmThreads), smem, stream, true, d_params, stages, kgroup, d_next, next_groups, two_prod);
    return cudaGetLastError();
}

}  // namespace tmae
