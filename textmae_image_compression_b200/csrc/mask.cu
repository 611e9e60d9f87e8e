// Score-guided patch ordering on the GPU: one CTA per image, everything in shared memory.
// Replaces the reference's host-side Python routine MCM.get_ids_shuffle (MCM.py:364-423, ~25 device->host syncs
// and 3-14 ms per sample) plus the index work of MCM.random_masking (MCM.py:579-583).
//
// The result must be bit-exact, and the routine is defined by fp32 ATen CPU kernels (quantile/lerp, cascade
// sum, softmax with Sleef expf, round-half-even), so this file restates that arithmetic operation by operation
// (see oracle/mask_oracle.c for the pinned CPU restatement).  COMPILED WITH -fmad=false: every fused
// multiply-add below is explicit.
#include <math.h>
#include <stdint.h>

#include "common.cuh"
#include "kernels.h"

namespace tmae {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int NQ = 9, NG = 10;

__device__ __forceinline__ float bits2f(uint32_t b) { return __uint_as_float(b); }
__device__ __forceinline__ int ceil_log2_i(int x) { int r = 0; while ((1 << r) < x) ++r; return r; }

// ATen lerp (native/Lerp.h), both arms contracted to one FMA by the CPU build.
__device__ __forceinline__ float lerp_aten(float lo, float hi, float w) {
    const float diff = __fsub_rn(hi, lo);
    if (fabsf(w) < 0.5f) return __fmaf_rn(w, diff, lo);
    return __fmaf_rn(-diff, __fsub_rn(1.0f, w), hi);
}

// Sleef_expf_u10 (FMA build) == ATen Vectorized<float>::exp used by the CPU softmax kernel.
__device__ __forceinline__ float exp_sleef_u10(float d) {
    const float R_LN2f = 1.442695040888963407359924681001892137426645954152985934135449406931f;
    const float L2Uf = 0.693145751953125f, L2Lf = 1.428606765330187045e-06f;
    const float qf = rintf(__fmul_rn(d, R_LN2f));
    const int q = (int)qf;
    float s = __fmaf_rn(qf, -L2Uf, d);
    s = __fmaf_rn(qf, -L2Lf, s);
    float u = 0.000198527617612853646278381f;
    u = __fmaf_rn(u, s, 0.00139304355252534151077271f);
    u = __fmaf_rn(u, s, 0.00833336077630519866943359f);
    u = __fmaf_rn(u, s, 0.0416664853692054748535156f);
    u = __fmaf_rn(u, s, 0.166666671633720397949219f);
    u = __fmaf_rn(u, s, 0.5f);
    u = __fadd_rn(1.0f, __fmaf_rn(__fmul_rn(s, s), u, s));
    const int q1 = q >> 1, q2 = q - q1;
    u = __fmul_rn(__fmul_rn(u, bits2f((uint32_t)(q1 + 127) << 23)), bits2f((uint32_t)(q2 + 127) << 23));
    if (d < -104.0f) u = 0.0f;
    if (d > 100.0f) u = INFINITY;
    return u;
}

__device__ __forceinline__ int float_to_int32_x86(float r) {       // cvttps2dq semantics
    if (isnan(r) || r >= 2147483648.0f || r < -2147483648.0f) return INT32_MIN;
    return (int)r;
}

// ATen cascade_sum (native/cpu/SumKernel.cpp) of n fp32 values with 8-lane vectors, cooperatively by one warp:
// lane = 8*row + vec_lane reproduces the 4 interleaved row accumulators of multi_row_sum.
__device__ float aten_sum_warp(const float* __restrict__ x, int n, int lane) {
    if (n >= 8) {
        const int vec_size = n >> 3, size_ilp = vec_size >> 2;
        int lp = ceil_log2_i(size_ilp) / 4;
        if (lp < 4) lp = 4;
        const int step = 1 << lp, lmask = step - 1;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        int i = 0;
        while (i + step <= size_ilp) {
            for (int j = 0; j < step; ++j, ++i) a0 = __fadd_rn(a0, x[i * 32 + lane]);
            a1 = __fadd_rn(a1, a0); a0 = 0.f;
            if ((i & (lmask << lp)) != 0) continue;
            a2 = __fadd_rn(a2, a1); a1 = 0.f;
            if ((i & (lmask << (2 * lp))) != 0) continue;
            a3 = __fadd_rn(a3, a2); a2 = 0.f;
        }
        for (; i < size_ilp; ++i) a0 = __fadd_rn(a0, x[i * 32 + lane]);
        a0 = __fadd_rn(a0, a1); a0 = __fadd_rn(a0, a2); a0 = __fadd_rn(a0, a3);
        for (int v = size_ilp * 4; v < vec_size; ++v)
            if (lane < 8) a0 = __fadd_rn(a0, x[v * 8 + lane]);
        const int l = lane & 7;
        const float r1 = __shfl_sync(0xffffffffu, a0, l + 8);
        const float r2 = __shfl_sync(0xffffffffu, a0, l + 16);
        const float r3 = __shfl_sync(0xffffffffu, a0, l + 24);
        float ps0 = __shfl_sync(0xffffffffu, a0, l);
        ps0 = __fadd_rn(ps0, r1); ps0 = __fadd_rn(ps0, r2); ps0 = __fadd_rn(ps0, r3);
        float fin = 0.f;
        for (int k = vec_size * 8; k < n; ++k) fin = __fadd_rn(fin, x[k]);
        for (int ll = 0; ll < 8; ++ll) fin = __fadd_rn(fin, __shfl_sync(0xffffffffu, ps0, ll));
        return __fadd_rn(0.0f, fin);
    }
    float ps[4] = {0.f, 0.f, 0.f, 0.f};
    const int size_ilp = n >> 2;
    for (int i = 0; i < size_ilp; ++i)
        for (int k = 0; k < 4; ++k) ps[k] = __fadd_rn(ps[k], x[i * 4 + k]);
    for (int i = size_ilp * 4; i < n; ++i) ps[0] = __fadd_rn(ps[0], x[i]);
    ps[0] = __fadd_rn(ps[0], ps[1]); ps[0] = __fadd_rn(ps[0], ps[2]); ps[0] = __fadd_rn(ps[0], ps[3]);
    return __fadd_rn(0.0f, ps[0]);
}

// Block-wide exclusive scan of an int array in shared memory (len <= 16 * kThreads); returns the total.
__device__ int block_exclusive_scan(int* a, int len, int* warp_tmp) {
    const int per = (len + kThreads - 1) / kThreads;
    const int beg = threadIdx.x * per;
    int local = 0;
    for (int i = 0; i < per; ++i) { const int p = beg + i; if (p < len) local += a[p]; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) warp_tmp[warp] = incl;
    __syncthreads();
    int woff = 0, total = 0;
    for (int w = 0; w < kWarps; ++w) { const int t = warp_tmp[w]; if (w < warp) woff += t; total += t; }
    int run = woff + incl - local;
    for (int i = 0; i < per; ++i) {
        const int p = beg + i;
        if (p < len) { const int t = a[p]; a[p] = run; run += t; }
    }
    __syncthreads();
    return total;
}

__global__ void __launch_bounds__(kThreads)
mask_select_kernel(const float* __restrict__ scores, int L, int Lp2, int K, int isa, int64_t* __restrict__ ids_shuffle,
                   int64_t* __restrict__ ids_restore, int64_t* __restrict__ ids_keep, const IoBlock* __restrict__ io) {
    pdl_launch_dependents();                     // first kernel of the forward (follows a memset): launched without PDL itself
    if (io) { scores = io->scores; ids_shuffle = io->out.ids_shuffle; ids_restore = io->out.ids_restore; }
    extern __shared__ float smf[];
    float* s = smf;                                   // scores in index order
    float* srt = s + Lp2;                             // ascending, +INF padded
    float* gvals = srt + Lp2;                         // unique values, later group-compacted values
    int* cat = reinterpret_cast<int*>(gvals + Lp2);
    int* first = cat + Lp2;                           // smallest index holding the same value
    int* pos = first + Lp2;                           // final position (or -1 while unselected)
    int* scan = pos + Lp2;                            // scratch for scans
    __shared__ float thr[NQ], means[NG];
    __shared__ int gsize[NG], goff[NG + 1], taken[NQ], base[NQ], warp_tmp[kWarps];
    __shared__ int sh_nu;

    const int n = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* sc = scores + (size_t)n * L;

    for (int i = tid; i < Lp2; i += kThreads) {
        const float v = i < L ? sc[i] : INFINITY;
        if (i < L) s[i] = v;
        srt[i] = v;
    }
    if (tid < NG) gsize[tid] = 0;
    __syncthreads();

    // ---- bitonic sort (ascending) ----
    for (int k = 2; k <= Lp2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < Lp2; i += kThreads) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const float a = srt[i], b = srt[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) { srt[i] = b; srt[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }

    // ---- unique(): MCM.py:384 ----
    for (int i = tid; i < Lp2; i += kThreads) scan[i] = (i < L && (i == 0 || srt[i] != srt[i - 1])) ? 1 : 0;
    __syncthreads();
    const int nu = block_exclusive_scan(scan, Lp2, warp_tmp);
    for (int i = tid; i < L; i += kThreads)
        if (i == 0 || srt[i] != srt[i - 1]) gvals[scan[i]] = srt[i];
    if (tid == 0) sh_nu = nu;
    __syncthreads();

    // ---- quantile(linear) thresholds: MCM.py:381-384 ----
    if (tid < NQ) {
        const uint32_t qbits[NQ] = {0x3dcccccdu, 0x3e4ccccdu, 0x3e99999au, 0x3ecccccdu, 0x3f000000u,
                                    0x3f19999au, 0x3f333333u, 0x3f4ccccdu, 0x3f666666u};
        const float rank = __fmul_rn(bits2f(qbits[tid]), (float)(nu - 1));
        const int below = (int)rank;
        const float w = __fsub_rn(rank, (float)below);
        const int above = (int)ceilf(rank);
        thr[tid] = lerp_aten(gvals[below], gvals[above], w);
    }
    __syncthreads();

    // ---- bucketize (right=False): MCM.py:387 ----
    for (int i = tid; i < L; i += kThreads) {
        const float v = s[i];
        int c = 0;
        while (c < NQ && thr[c] < v) ++c;
        cat[i] = c;
        atomicAdd(&gsize[c], 1);
    }
    __syncthreads();
    if (tid == 0) {
        int o = 0;
        for (int g = 0; g < NG; ++g) { goff[g] = o; o += gsize[g]; }
        goff[NG] = o;
    }
    __syncthreads();

    // ---- per-group values in index order, then ATen mean: MCM.py:390-393 ----
    for (int g = warp; g < NG; g += kWarps) {
        int run = goff[g];
        for (int i0 = 0; i0 < L; i0 += 32) {
            const int i = i0 + lane;
            const bool in = i < L && cat[i] == g;
            const unsigned m = __ballot_sync(0xffffffffu, in);
            if (in) gvals[run + __popc(m & ((1u << lane) - 1u))] = s[i];
            run += __popc(m);
        }
    }
    __syncthreads();
    for (int g = warp; g < NG; g += kWarps) {
        const int m = gsize[g];
        const float sum = aten_sum_warp(gvals + goff[g], m, lane);
        if (lane == 0) means[g] = __fdiv_rn(sum, (float)m);          // 0/0 = NaN for an empty group
    }
    __syncthreads();

    // ---- softmax over the 9 lower groups, rounded counts, Python-slice take counts: MCM.py:399-408 ----
    if (tid == 0) {
        float mx = means[0];
        bool has_nan = isnan(means[0]);
        for (int i = 1; i < NQ; ++i) { if (isnan(means[i])) has_nan = true; if (means[i] > mx) mx = means[i]; }
        float sm[NQ];
        if (has_nan) {
            for (int i = 0; i < NQ; ++i) sm[i] = NAN;
        } else {
            float e[NQ];
            for (int i = 0; i < NQ; ++i) e[i] = exp_sleef_u10(__fsub_rn(means[i], mx));
            float sum;
            if (isa == 16) {
                sum = e[0];
                for (int i = 1; i < NQ; ++i) sum = __fadd_rn(sum, e[i]);
            } else {
                const float l0 = __fadd_rn(e[0], e[8]);
                const float a0 = __fadd_rn(l0, e[4]), a1 = __fadd_rn(e[1], e[5]);
                const float a2 = __fadd_rn(e[2], e[6]), a3 = __fadd_rn(e[3], e[7]);
                sum = __fadd_rn(__fadd_rn(a0, a2), __fadd_rn(a1, a3));
            }
            const float rcp = __fdiv_rn(1.0f, sum);
            for (int i = 0; i < NQ; ++i) sm[i] = __fmul_rn(e[i], rcp);
        }
        const int n_top = gsize[9];
        const int new_target = K - n_top;
        int acc = n_top;
        for (int g = 0; g < NQ; ++g) {
            const int cnt = float_to_int32_x86(rintf(__fmul_rn(sm[g], (float)new_target)));
            const int m = gsize[g];
            const int32_t start = (int32_t)((uint32_t)m - (uint32_t)cnt);     // int32 wrap-around
            long long st = start;
            if (st < 0) { st += m; if (st < 0) st = 0; }                      // Python slice semantics
            if (st > m) st = m;
            taken[g] = m - (int)st;
            base[g] = acc;
            acc += taken[g];
        }
    }
    __syncthreads();

    // ---- first-equal index and rank among equal values ----
    for (int i = tid; i < L; i += kThreads) {
        const float v = s[i];
        int eqb = 0, fi = i;
        for (int j = 0; j < i; ++j)
            if (s[j] == v) { if (eqb == 0) fi = j; ++eqb; }
        first[i] = fi;
        const int g = cat[i];
        int p = -1;
        if (g < 9) {
            int lo = 0, hi = L;                                   // lower_bound
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (srt[mid] < v) lo = mid + 1; else hi = mid; }
            const int lower = lo;
            hi = L;                                               // upper_bound
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (srt[mid] <= v) lo = mid + 1; else hi = mid; }
            const int upper = lo;
            const int a = lower - goff[g], b = upper - goff[g];
            const int cut = gsize[g] - taken[g];
            const int from = a > cut ? a : cut;
            const int freq = b - from;
            if (eqb < freq) p = base[g] + (from - cut) + eqb;
        } else {
            p = -2 - eqb;                                         // resolved below (needs every first[])
        }
        pos[i] = p;
    }
    __syncthreads();
    // top decile: Counter() first-appearance order of values, then index order within a value (MCM.py:396,410-416)
    for (int i = tid; i < L; i += kThreads) {
        if (cat[i] != 9) continue;
        const int fi = first[i];
        int before = 0;
        for (int j = 0; j < L; ++j) before += (cat[j] == 9 && first[j] < fi) ? 1 : 0;
        pos[i] = before + (-2 - pos[i]);
    }
    __syncthreads();

    // ---- unselected indices ascending: MCM.py:418-420 ----
    // They follow the selected ones.  A NaN score equals no value (MCM.py:410-416 selects nothing for it), so a row of NaN scores
    // (0/0 of a flat image) selects fewer indices than the take counts add up to: ids 0, 1, 2, ... for an all-NaN row.
    for (int i = tid; i < Lp2; i += kThreads) scan[i] = (i < L && pos[i] == -1) ? 1 : 0;
    __syncthreads();
    const int total_sel = L - block_exclusive_scan(scan, Lp2, warp_tmp);
    for (int i = tid; i < L; i += kThreads) {
        const int p = pos[i] == -1 ? total_sel + scan[i] : pos[i];
        if (ids_shuffle) ids_shuffle[(size_t)n * L + p] = i;
        if (ids_restore) ids_restore[(size_t)n * L + i] = p;
        if (ids_keep && p < K) ids_keep[(size_t)n * K + p] = i;
    }
}

}  // namespace

cudaError_t launch_mask_select(const float* scores, int N, int L, int K, int softmax_isa, int64_t* ids_shuffle,
                               int64_t* ids_restore, int64_t* ids_keep, cudaStream_t st, const IoBlock* io) {
    if (N == 0) return cudaSuccess;
    int Lp2 = 32;
    while (Lp2 < L) Lp2 <<= 1;
    if (Lp2 > 16 * kThreads) return cudaErrorInvalidValue;
    const size_t smem = (size_t)Lp2 * 7 * sizeof(float);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(mask_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    TMAE_CARVEOUT_ONCE(mask_select_kernel);
    mask_select_kernel<<<N, kThreads, smem, st>>>(scores, L, Lp2, K, softmax_isa == 8 ? 8 : 16, ids_shuffle,
                                                  ids_restore, ids_keep, io);
    return cudaGetLastError();
}

}  // namespace tmae
