// HBM-bound kernels of the path: kept-patch gather (im2col), LayerNorm, the entropy-model elementwise work
// (factorized-prior and Gaussian likelihoods, quantisation, log2-rate reduction) and weight prepacking.
// All are coalesced, 128-bit vectorised where the layout allows, with warp-shuffle reductions.
#include <math.h>

#include "common.cuh"
#include "kernels.h"

namespace tmae {

// ---------------------------------------------------------------------------------------------------------
// Kept-patch gather: timm PatchEmbed's im2col restricted to the K kept patches (MCM.py:615 + :583-586; the
// conv is a per-patch linear map, so gathering first is row-wise identical).  Row (n, j) of `patches` holds
// patch ids_keep[n, j] flattened in (c, p, q) order == Conv2d weight order.  Block (n, j == K) writes the cls row
// x[n*T + 0] = cls_token + pos_embed[0] (MCM.py:624-626).
// grid (K + 1, N), block 192: thread = (c, p, q4) handles 4 pixels (16 B read, 8 B write).
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(192)
gather_patches_kernel(const float* __restrict__ imgs, const int64_t* __restrict__ ids_keep,
                      __nv_bfloat16* __restrict__ patches, float* __restrict__ x, const float* __restrict__ cls_token,
                      const float* __restrict__ pos_embed, int S, int grid_w, int K, int T, int C, int in_chans,
                      int patch, long long lo_off, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    if (io) imgs = io->imgs;
    const int j = blockIdx.x, n = blockIdx.y;
    if (j == K) {
        float* dst = x + (size_t)n * T * C;
        for (int c = threadIdx.x; c < C; c += blockDim.x) dst[c] = cls_token[c] + pos_embed[c];
        return;
    }
    const int pid = (int)ids_keep[(size_t)n * K + j];
    const int py = pid / grid_w, px = pid - py * grid_w;
    const int per_c = patch * patch;               // 256
    const int row_len = in_chans * per_c;          // 768
    __nv_bfloat16* dst = patches + ((size_t)n * K + j) * row_len;
    for (int e = threadIdx.x * 4; e < row_len; e += blockDim.x * 4) {
        const int c = e / per_c;
        const int rem = e - c * per_c;
        const int p = rem / patch, q = rem - p * patch;
        const float4 v = __ldg(reinterpret_cast<const float4*>(
            imgs + (((size_t)n * in_chans + c) * S + (py * patch + p)) * S + px * patch + q));
        store_bf16x4_planes(dst + e, lo_off, v.x, v.y, v.z, v.w);     // precise patch embed: extra planes of the residual
    }
}

cudaError_t launch_gather_patches(const float* imgs, const int64_t* ids_keep, __nv_bfloat16* patches, float* x,
                                  const float* cls_token, const float* pos_embed, int N, int S, int grid_w, int K,
                                  int T, int C, int in_chans, int patch, long long lo_off, cudaStream_t st, const IoBlock* io) {
    dim3 grid(K + 1, N);
    TMAE_CARVEOUT_ONCE(gather_patches_kernel);
    return launch_k(gather_patches_kernel, grid, dim3(192), 0, st, true, imgs, ids_keep, patches, x, cls_token, pos_embed, S,
                    grid_w, K, T, C, in_chans, patch, lo_off, io);
}

// ---------------------------------------------------------------------------------------------------------
// LayerNorm (eps 1e-6, MCM.py:46): fp32 residual row in, bf16 normalised row out.  One warp per row, the row is
// held in registers (C <= 1024 * ... via float4), two-pass mean / centred variance like ATen.
// drop_cls = 1: the final encoder_norm (MCM.py:631-632) skips token 0 and writes compact rows n*K + (t-1);
// optionally also fp32 (x_remain output).
// ---------------------------------------------------------------------------------------------------------
template <int VEC_PER_LANE>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                 __nv_bfloat16* __restrict__ out, float* __restrict__ out_f32, int rows, int C, int T, int drop_cls,
                 float eps, long long lo_off, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    if (io) out_f32 = io->out.x_remain;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= rows) return;
    long long orow = warp;
    if (drop_cls) {
        const int n = warp / T, t = warp - n * T;
        if (t == 0) return;
        orow = (long long)n * (T - 1) + (t - 1);
    }
    const float4* src = reinterpret_cast<const float4*>(x + (size_t)warp * C);
    float4 v[VEC_PER_LANE];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < VEC_PER_LANE; ++i) {
        v[i] = src[i * 32 + lane];
        sum += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    const float mean = warp_sum(sum) / (float)C;
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < VEC_PER_LANE; ++i) {
        const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
        sq += a * a + b * b + c * c + d * d;
    }
    const float rstd = rsqrtf(warp_sum(sq) / (float)C + eps);
    const float4* g4 = reinterpret_cast<const float4*>(gamma);
    const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
    for (int i = 0; i < VEC_PER_LANE; ++i) {
        const float4 g = __ldg(g4 + i * 32 + lane), b = __ldg(b4 + i * 32 + lane);
        const float o0 = (v[i].x - mean) * rstd * g.x + b.x;
        const float o1 = (v[i].y - mean) * rstd * g.y + b.y;
        const float o2 = (v[i].z - mean) * rstd * g.z + b.z;
        const float o3 = (v[i].w - mean) * rstd * g.w + b.w;
        __nv_bfloat16* dst = out + (size_t)orow * C + (i * 32 + lane) * 4;
        store_bf16x4_planes(dst, lo_off, o0, o1, o2, o3);             // extra planes when the consumer is a precise layer
        if (out_f32) *reinterpret_cast<float4*>(out_f32 + (size_t)orow * C + (i * 32 + lane) * 4) = make_float4(o0, o1, o2, o3);
    }
}

cudaError_t launch_layernorm(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out, float* out_f32,
                             int rows, int C, int T, int drop_cls, float eps, long long lo_off, cudaStream_t st, const IoBlock* io) {
    const int blocks = (rows * 32 + 255) / 256;
    if (C % 128 != 0) return cudaErrorInvalidValue;
    switch (C / 128) {
        case 6: TMAE_CARVEOUT_ONCE(layernorm_kernel<6>); return launch_k(layernorm_kernel<6>, dim3(blocks), dim3(256), 0, st, true, x, gamma, beta, out, out_f32, rows, C, T, drop_cls, eps, lo_off, io);
        case 8: TMAE_CARVEOUT_ONCE(layernorm_kernel<8>); return launch_k(layernorm_kernel<8>, dim3(blocks), dim3(256), 0, st, true, x, gamma, beta, out, out_f32, rows, C, T, drop_cls, eps, lo_off, io);
        case 10: TMAE_CARVEOUT_ONCE(layernorm_kernel<10>); return launch_k(layernorm_kernel<10>, dim3(blocks), dim3(256), 0, st, true, x, gamma, beta, out, out_f32, rows, C, T, drop_cls, eps, lo_off, io);
        case 1: TMAE_CARVEOUT_ONCE(layernorm_kernel<1>); return launch_k(layernorm_kernel<1>, dim3(blocks), dim3(256), 0, st, true, x, gamma, beta, out, out_f32, rows, C, T, drop_cls, eps, lo_off, io);
        case 2: TMAE_CARVEOUT_ONCE(layernorm_kernel<2>); return launch_k(layernorm_kernel<2>, dim3(blocks), dim3(256), 0, st, true, x, gamma, beta, out, out_f32, rows, C, T, drop_cls, eps, lo_off, io);
        case 3: TMAE_CARVEOUT_ONCE(layernorm_kernel<3>); return launch_k(layernorm_kernel<3>, dim3(blocks), dim3(256), 0, st, true, x, gamma, beta, out, out_f32, rows, C, T, drop_cls, eps, lo_off, io);
        case 4: TMAE_CARVEOUT_ONCE(layernorm_kernel<4>); return launch_k(layernorm_kernel<4>, dim3(blocks), dim3(256), 0, st, true, x, gamma, beta, out, out_f32, rows, C, T, drop_cls, eps, lo_off, io);
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// Factorized-prior likelihood of z + quantisation (compressai EntropyBottleneck eval forward, MCM.py:741-744).
// eb_tab: [64][Cz] fp32, parameter-major (coalesced across channels); per channel the 64 entries are: softplus(matrix0)[3] bias0[3] tanh(factor0)[3] | softplus(matrix1)[9] bias1[3]
// tanh(factor1)[3] | (x2 more 3x3 layers) | softplus(matrix4)[3] bias4[1] | median at [60].
// ---------------------------------------------------------------------------------------------------------
// t: this channel's column of the parameter-major table (entry k at t[k * cs], cs = Cz): consecutive lanes handle
// consecutive channels, so every table read of a warp is one coalesced 128-byte line.
__device__ __forceinline__ float eb_logits(const float* __restrict__ t, int cs, float x) {
    float h[3], g[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        float v = t[i * cs] * x + t[(3 + i) * cs];
        h[i] = v + t[(6 + i) * cs] * tanhf(v);
    }
    const float* tt = t + 9 * cs;
#pragma unroll
    for (int l = 0; l < 3; ++l) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            float v = tt[(i * 3 + 0) * cs] * h[0];
            v += tt[(i * 3 + 1) * cs] * h[1];
            v += tt[(i * 3 + 2) * cs] * h[2];
            v += tt[(9 + i) * cs];
            g[i] = v + tt[(12 + i) * cs] * tanhf(v);
        }
        h[0] = g[0]; h[1] = g[1]; h[2] = g[2];
        tt += 15 * cs;
    }
    float v = tt[0] * h[0];
    v += tt[1 * cs] * h[1];
    v += tt[2 * cs] * h[2];
    return v + tt[3 * cs];
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// z: [rows, Cz] compact channels-last.  zhat_bf (optional): bf16 copy, same layout, the input of h_s.
__global__ void __launch_bounds__(256)
bottleneck_kernel(const float* __restrict__ z, const float* __restrict__ eb_tab, long long total, int Cz,
                  float* __restrict__ lik_out, int32_t* __restrict__ sym_out, float* __restrict__ zhat_out,
                  __nv_bfloat16* __restrict__ zhat_bf, long long lo_off, int s4, double* __restrict__ rate_acc, int rows_per_image,
                  int16_t* __restrict__ sym16_out, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    if (io) { lik_out = io->out.z_likelihoods; sym_out = io->out.z_symbols; zhat_out = io->out.z_hat; sym16_out = io->out.z_symbols_i16; }
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float lg = 0.f;
    int n = 0;
    if (idx < total) {
        const long long row = idx / Cz;
        const int c = (int)(idx - row * Cz);
        const float* t = eb_tab + c;
        const float med = t[60 * Cz];
        const float sym = rintf(z[idx] - med);
        const float zh = sym + med;
        const float lower = eb_logits(t, Cz, zh - 0.5f);
        const float upper = eb_logits(t, Cz, zh + 0.5f);
        const float sum = lower + upper;
        const float sgn = sum > 0.f ? -1.f : (sum < 0.f ? 1.f : 0.f);
        float lik = fabsf(sigmoidf_(sgn * upper) - sigmoidf_(sgn * lower));
        lik = fmaxf(lik, 1e-9f);
        if (lik_out) lik_out[idx] = lik;
        if (sym_out) sym_out[idx] = (int32_t)sym;
        if (sym16_out) sym16_out[idx] = (int16_t)fminf(fmaxf(sym, -32768.f), 32767.f);
        if (zhat_out) zhat_out[idx] = zh;
        n = (int)(row / rows_per_image);
        if (zhat_bf) store_bf16_planes(zhat_bf + idx, lo_off, zh);
        lg = log2f(lik);
    }
    if (rate_acc) {
        // a warp may straddle two images when Cz*rows_per_image is not a multiple of 32: reduce per image id
        const int n0 = __shfl_sync(0xffffffffu, n, 0);
        const bool same = __all_sync(0xffffffffu, (idx >= total) || n == n0);
        if (same) {
            const float s = warp_sum(lg);
            if ((threadIdx.x & 31) == 0 && s != 0.f) atomicAdd(rate_acc + n0, (double)s);
        } else if (idx < total) {
            atomicAdd(rate_acc + n, (double)lg);
        }
    }
}

cudaError_t launch_bottleneck(const float* z, const float* eb_tab, long long rows, int Cz, float* lik, int32_t* sym,
                              float* zhat, __nv_bfloat16* zhat_bf, long long lo_off, int s4, double* rate_acc, int rows_per_image,
                              int16_t* sym16, cudaStream_t st, const IoBlock* io) {
    const long long total = rows * Cz;
    if (total == 0) return cudaSuccess;
    const int blocks = (int)((total + 255) / 256);
    TMAE_CARVEOUT_ONCE(bottleneck_kernel);
    return launch_k(bottleneck_kernel, dim3(blocks), dim3(256), 0, st, true, z, eb_tab, total, Cz, lik, sym, zhat, zhat_bf, lo_off, s4,
                    rate_acc, rows_per_image, sym16, io);
}

// ---------------------------------------------------------------------------------------------------------
// Gaussian conditional likelihood + quantisation of one latent slice (compressai GaussianConditional eval
// forward + quantize_ste, MCM.py:771-776).  Each thread handles 4 consecutive channels (128-bit accesses).
//   y, mu, sigma, lik, sym, y_hat : fp32 / int32 [rows, ld] with channel offset col0, `cs` channels in the slice.
//   yhat_bf (optional) : bf16 copy [rows, ld_bf], same channel offset: support for later slices.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gaussian_slice_kernel(const float* __restrict__ y, const float* __restrict__ mu, const float* __restrict__ sigma,
                      long long rows, int ld, int col0, int cs, float* __restrict__ lik_out,
                      int32_t* __restrict__ sym_out, float* __restrict__ yhat_out, __nv_bfloat16* __restrict__ yhat_bf,
                      long long lo_off, int ld_bf, int s, double* __restrict__ rate_acc, const float* __restrict__ scale_table,
                      int n_table, int16_t* __restrict__ sym16_out, int32_t* __restrict__ idx_out, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    if (io) { lik_out = io->out.y_likelihoods; sym_out = io->out.y_symbols; sym16_out = io->out.y_symbols_i16; idx_out = io->out.y_indexes; }
    const int vec_per_row = cs >> 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = rows * vec_per_row;
    float lg = 0.f;
    int n = 0;
    if (idx < total) {
        const long long row = idx / vec_per_row;
        const int c = col0 + (int)(idx - row * vec_per_row) * 4;
        const size_t off = (size_t)row * ld + c;
        const float4 yv = *reinterpret_cast<const float4*>(y + off);
        const float4 mv = *reinterpret_cast<const float4*>(mu + off);
        const float4 sv = *reinterpret_cast<const float4*>(sigma + off);
        float4 lk, sy, yh;
        gaussian_elem(yv.x, mv.x, sv.x, lk.x, sy.x, yh.x);
        gaussian_elem(yv.y, mv.y, sv.y, lk.y, sy.y, yh.y);
        gaussian_elem(yv.z, mv.z, sv.z, lk.z, sy.z, yh.z);
        gaussian_elem(yv.w, mv.w, sv.w, lk.w, sy.w, yh.w);
        if (lik_out) *reinterpret_cast<float4*>(lik_out + off) = lk;
        if (sym_out) *reinterpret_cast<int4*>(sym_out + off) = make_int4((int)sy.x, (int)sy.y, (int)sy.z, (int)sy.w);
        if (sym16_out) {
            auto sat = [](float v) { return (int16_t)fminf(fmaxf(v, -32768.f), 32767.f); };
            short4 s4v;
            s4v.x = sat(sy.x); s4v.y = sat(sy.y); s4v.z = sat(sy.z); s4v.w = sat(sy.w);
            *reinterpret_cast<short4*>(sym16_out + off) = s4v;
        }
        if (idx_out && scale_table) *reinterpret_cast<int4*>(idx_out + off) = scale_indexes4(scale_table, n_table, sv);
        if (yhat_out) *reinterpret_cast<float4*>(yhat_out + off) = yh;
        const int K = s * s;
        n = (int)(row / K);
        if (yhat_bf) {
            __nv_bfloat16* dst = yhat_bf + (size_t)row * ld_bf + c;
            store_bf16x4_planes(dst, lo_off, yh.x, yh.y, yh.z, yh.w);
        }
        lg = (log2f(lk.x) + log2f(lk.y)) + (log2f(lk.z) + log2f(lk.w));
    }
    if (rate_acc) {
        const int n0 = __shfl_sync(0xffffffffu, n, 0);
        const bool same = __all_sync(0xffffffffu, (idx >= total) || n == n0);
        if (same) {
            const float sm = warp_sum(lg);
            if ((threadIdx.x & 31) == 0 && sm != 0.f) atomicAdd(rate_acc + n0, (double)sm);
        } else if (idx < total) {
            atomicAdd(rate_acc + n, (double)lg);
        }
    }
}

cudaError_t launch_gaussian_slice(const float* y, const float* mu, const float* sigma, long long rows, int ld, int col0,
                                  int cs, float* lik, int32_t* sym, float* yhat, __nv_bfloat16* yhat_bf, long long lo_off,
                                  int ld_bf, int s, double* rate_acc, const float* scale_table, int n_table, int16_t* sym16,
                                  int32_t* idx, cudaStream_t st, const IoBlock* io) {
    const long long total = rows * (cs / 4);
    if (total == 0) return cudaSuccess;
    const int blocks = (int)((total + 255) / 256);
    TMAE_CARVEOUT_ONCE(gaussian_slice_kernel);
    return launch_k(gaussian_slice_kernel, dim3(blocks), dim3(256), 0, st, true, y, mu, sigma, rows, ld, col0, cs, lik, sym, yhat,
                    yhat_bf, lo_off, ld_bf, s, rate_acc, scale_table, n_table, sym16, idx, io);
}

// flat variant for the stand-alone operator (n elements, no layout)
__global__ void gaussian_flat_kernel(const float* __restrict__ y, const float* __restrict__ mu,
                                     const float* __restrict__ sigma, long long n, float* __restrict__ lik,
                                     int32_t* __restrict__ sym, float* __restrict__ yhat) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float l, s, h;
    gaussian_elem(y[i], mu[i], sigma[i], l, s, h);
    if (lik) lik[i] = l;
    if (sym) sym[i] = (int32_t)s;
    if (yhat) yhat[i] = h;
}
cudaError_t launch_gaussian_flat(const float* y, const float* mu, const float* sigma, long long n, float* lik,
                                 int32_t* sym, float* yhat, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    gaussian_flat_kernel<<<(int)((n + 255) / 256), 256, 0, st>>>(y, mu, sigma, n, lik, sym, yhat);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// Decode side (MCM.decompress, MCM.py:896-968, with the range decoder's symbols given): the symbols arrive in the range
// coder's order (per image, channel-major (c, y, x)), the latents stay channels-last like everywhere else.  The arithmetic
// is exactly the encoder's dequantisation - bottleneck_kernel's zh = sym + med and gaussian_elem's yhat = sym + mu - so a
// decoder of the same configuration reproduces the encoder's latents bit for bit.
// ---------------------------------------------------------------------------------------------------------
// z_hat = (float)sym + median (row 60 of eb_tab): fp32 to io->out.z_hat (optional) and the bf16 planes h_s reads.
__global__ void __launch_bounds__(256)
z_dequantize_kernel(const float* __restrict__ eb_tab, long long total, int Cz, int hw, __nv_bfloat16* __restrict__ zhat_bf,
                    long long lo_off, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long row = idx / Cz;
    const int c = (int)(idx - row * Cz);
    const long long n = row / hw;
    const int p = (int)(row - n * hw);
    const float zh = (float)io->z_symbols[(n * Cz + c) * hw + p] + eb_tab[60 * Cz + c];
    if (io->out.z_hat) io->out.z_hat[idx] = zh;
    store_bf16_planes(zhat_bf + idx, lo_off, zh);
}
cudaError_t launch_z_dequantize(const float* eb_tab, long long rows, int Cz, int hw, __nv_bfloat16* zhat_bf, long long lo_off,
                                cudaStream_t st, const IoBlock* io) {
    const long long total = rows * Cz;
    if (total == 0) return cudaSuccess;
    TMAE_CARVEOUT_ONCE(z_dequantize_kernel);
    return launch_k(z_dequantize_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, true, eb_tab, total, Cz, hw, zhat_bf,
                    lo_off, io);
}

// Scale-table indexes of `cs` channels from col0 of sigma [rows, ld] (the separate-GEMM path; the fused cc.8 layer emits
// them in its store phase) into io->out.y_indexes in the range coder's order.  Thread = 4 channels of one pixel.
__global__ void __launch_bounds__(256)
slice_indexes_kernel(const float* __restrict__ sigma, long long rows, int ld, int col0, int cs, int hw, const float* __restrict__ scale_table,
                     int n_table, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    const int vec_per_row = cs >> 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * vec_per_row) return;
    const long long row = idx / vec_per_row;
    const int c = col0 + (int)(idx - row * vec_per_row) * 4;
    const long long n = row / hw;
    const int p = (int)(row - n * hw);
    const int4 id = scale_indexes4(scale_table, n_table, *reinterpret_cast<const float4*>(sigma + (size_t)row * ld + c));
    int32_t* dst = io->out.y_indexes + (n * ld + c) * hw + p;
    dst[0] = id.x; dst[hw] = id.y; dst[2 * hw] = id.z; dst[3 * hw] = id.w;
}
cudaError_t launch_slice_indexes(const float* sigma, long long rows, int ld, int col0, int cs, int hw, const float* scale_table,
                                 int n_table, cudaStream_t st, const IoBlock* io) {
    const long long total = rows * (cs / 4);
    if (total == 0) return cudaSuccess;
    TMAE_CARVEOUT_ONCE(slice_indexes_kernel);
    return launch_k(slice_indexes_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, true, sigma, rows, ld, col0, cs, hw,
                    scale_table, n_table, io);
}

// y_hat = (float)sym + mu for `cs` channels from col0: the caller's symbols (io->y_symbols, range-coder order) and this
// run's mu -> fp32 yhat [rows, ld] and its bf16 planes (support of the later slices; LRP then adds in place, as in the
// forward).  Thread = 4 channels of one pixel.
__global__ void __launch_bounds__(256)
slice_dequantize_kernel(const float* __restrict__ mu, long long rows, int ld, int col0, int cs, int hw, float* __restrict__ yhat,
                        __nv_bfloat16* __restrict__ yhat_bf, long long lo_off, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    const int vec_per_row = cs >> 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * vec_per_row) return;
    const long long row = idx / vec_per_row;
    const int c = col0 + (int)(idx - row * vec_per_row) * 4;
    const long long n = row / hw;
    const int p = (int)(row - n * hw);
    const int32_t* sym = io->y_symbols + (n * ld + c) * hw + p;
    const size_t off = (size_t)row * ld + c;
    const float4 mv = *reinterpret_cast<const float4*>(mu + off);
    const float4 yh = make_float4((float)sym[0] + mv.x, (float)sym[hw] + mv.y, (float)sym[2 * hw] + mv.z, (float)sym[3 * hw] + mv.w);
    *reinterpret_cast<float4*>(yhat + off) = yh;
    store_bf16x4_planes(yhat_bf + off, lo_off, yh.x, yh.y, yh.z, yh.w);
}
cudaError_t launch_slice_dequantize(const float* mu, long long rows, int ld, int col0, int cs, int hw, float* yhat,
                                    __nv_bfloat16* yhat_bf, long long lo_off, cudaStream_t st, const IoBlock* io) {
    const long long total = rows * (cs / 4);
    if (total == 0) return cudaSuccess;
    TMAE_CARVEOUT_ONCE(slice_dequantize_kernel);
    return launch_k(slice_dequantize_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, true, mu, rows, ld, col0, cs, hw,
                    yhat, yhat_bf, lo_off, io);
}

// ---------------------------------------------------------------------------------------------------------
// Rate finalise:bpp[n] = -sum(log2 lik) / S^2 (rd_loss.py:15-20, per image) and the batch pair
// {sum log2 lik, N*S*S} that the data-parallel all-reduce combines.
// ---------------------------------------------------------------------------------------------------------
__global__ void rate_finalize_kernel(const double* __restrict__ rate_acc, int N, double pixels_per_image,
                                     float* __restrict__ bpp, double* __restrict__ rate_sums,
                                     const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    if (io) {                                  // caller buffers when given, else the workspace defaults passed in
        if (io->out.bpp) bpp = io->out.bpp;
        if (io->out.rate_sums) rate_sums = io->out.rate_sums;
    }
    double tot = 0.0;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        const double a = rate_acc[n];
        if (bpp) bpp[n] = (float)(-a / pixels_per_image);
        tot += a;
    }
    __shared__ double sh[32];
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = tot;
    __syncthreads();
    if (threadIdx.x == 0 && rate_sums) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
        rate_sums[0] = t;
        rate_sums[1] = pixels_per_image * N;
    }
}
cudaError_t launch_rate_finalize(const double* rate_acc, int N, double pixels_per_image, float* bpp,
                                 double* rate_sums, cudaStream_t st, const IoBlock* io) {
    TMAE_CARVEOUT_ONCE(rate_finalize_kernel);
    return launch_k(rate_finalize_kernel, dim3(1), dim3(256), 0, st, true, rate_acc, N, pixels_per_image, bpp, rate_sums, io);
}

// ---------------------------------------------------------------------------------------------------------
// Optional copies of workspace-resident results into the caller's buffers (pointers read from the IoBlock).
// ---------------------------------------------------------------------------------------------------------
__global__ void copy_outputs_kernel(const IoBlock* __restrict__ io, const float4* __restrict__ y, const float4* __restrict__ z,
                                    const float4* __restrict__ mu, const float4* __restrict__ sigma,
                                    const float4* __restrict__ yhat, const int64_t* __restrict__ ids_keep, long long n_y4,
                                    long long n_z4, long long n_ids) {
    pdl_wait();
    pdl_launch_dependents();
    const tmae_outputs o = io->out;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_y4; i += stride) {
        if (o.y) reinterpret_cast<float4*>(o.y)[i] = y[i];
        if (o.mu) reinterpret_cast<float4*>(o.mu)[i] = mu[i];
        if (o.sigma) reinterpret_cast<float4*>(o.sigma)[i] = sigma[i];
        if (o.y_hat) reinterpret_cast<float4*>(o.y_hat)[i] = yhat[i];
        if (i < n_z4 && o.z) reinterpret_cast<float4*>(o.z)[i] = z[i];
        if (i < n_ids && o.ids_keep) o.ids_keep[i] = ids_keep[i];
    }
}
cudaError_t launch_copy_outputs(const IoBlock* io, const float* y, const float* z, const float* mu, const float* sigma,
                                const float* yhat, const int64_t* ids_keep, long long n_y, long long n_z, long long n_ids,
                                cudaStream_t st) {
    TMAE_CARVEOUT_ONCE(copy_outputs_kernel);
    return launch_k(copy_outputs_kernel, dim3(296), dim3(256), 0, st, true, io, reinterpret_cast<const float4*>(y),
                    reinterpret_cast<const float4*>(z), reinterpret_cast<const float4*>(mu), reinterpret_cast<const float4*>(sigma),
                    reinterpret_cast<const float4*>(yhat), ids_keep, n_y / 4, n_z / 4, n_ids);
}


// ---------------------------------------------------------------------------------------------------------
// Symbol / index packing for the entropy coder (SURVEY 8f-1): the reference hands `encode_with_indexes` the symbols of
// slice 0, 1, ... each flattened in (c, y, x) order (MCM.py:867-873) == the NCHW order of the whole [Cy, s, s] latent of
// an image.  The path keeps everything channels-last, so this transposes [N, hw, C] -> [N, C, hw] through a 32x32 tile.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pack_nchw_i32_kernel(const int32_t* __restrict__ src, int32_t* __restrict__ dst, int hw, int C) {
    __shared__ int32_t tile[32][33];
    const int n = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int32_t* s = src + (size_t)n * hw * C;
    int32_t* d = dst + (size_t)n * hw * C;
    for (int r = ty; r < 32; r += 8)
        if (p0 + r < hw && c0 + tx < C) tile[r][tx] = s[(size_t)(p0 + r) * C + c0 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8)
        if (c0 + r < C && p0 + tx < hw) d[(size_t)(c0 + r) * hw + p0 + tx] = tile[tx][r];
}
cudaError_t launch_pack_nchw_i32(const int32_t* src, int32_t* dst, int N, int hw, int C, cudaStream_t st) {
    if (N == 0) return cudaSuccess;
    dim3 grid((hw + 31) / 32, (C + 31) / 32, N);
    pack_nchw_i32_kernel<<<grid, 256, 0, st>>>(src, dst, hw, C);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// Weight prepack: fp32 [Cout, Cin_total, kh, kw] (or [Cout, Cin] linear) -> bf16 [Cout, Kp], K index =
// tap-major, then channel segment (each padded to a multiple of 64 with zeros), then channel.
// shuffle = 1: output row q*Cq + c takes source channel c*4 + q (PixelShuffle(2) made contiguous per quadrant).
// planes = 2 / 3 (precise layers): every tap holds its segments once per plane - the hi planes bf16(w), then
// bf16(w - hi) (and bf16(w - hi - mid) for the three-plane / fp32-exact form).
// ---------------------------------------------------------------------------------------------------------
__global__ void prepack_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int Cout,
                                      int Cin_total, int taps, int nseg, int seg_c0, int seg_c1, int seg_c2,
                                      int shuffle, int planes, const float* __restrict__ gamma) {
    const int segc[3] = {seg_c0, seg_c1, seg_c2};
    int segpad[3], kp_tap = 0;
    for (int i = 0; i < 3; ++i) {
        segpad[i] = i < nseg ? ((segc[i] + 63) / 64) * 64 : 0;
        kp_tap += segpad[i];
    }
    const long long Kp = (long long)kp_tap * taps * planes;
    const long long total = (long long)Cout * Kp;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int ro = (int)(idx / Kp);
        const long long kidx = idx - (long long)ro * Kp;
        const int tap = (int)(kidx / (kp_tap * planes));
        int within = (int)(kidx - (long long)tap * kp_tap * planes);
        const int plane = within / kp_tap;
        within -= plane * kp_tap;
        int ci = -1, cbase = 0;
        for (int i = 0; i < nseg; ++i) {
            if (within < segpad[i]) {
                if (within < segc[i]) ci = cbase + within;
                break;
            }
            within -= segpad[i];
            cbase += segc[i];
        }
        int co = ro;
        if (shuffle) {
            const int cq = Cout >> 2;
            const int q = ro / cq, c = ro - q * cq;
            co = c * 4 + q;
        }
        float v = 0.f;
        if (ci >= 0) v = w[((size_t)co * Cin_total + ci) * taps + tap];
        if (ci >= 0 && gamma != nullptr) v *= gamma[ci];          // LayerNorm folded into this linear: W' = W diag(gamma)
        const __nv_bfloat16 hi = __float2bfloat16(v);
        const float r1 = v - __bfloat162float(hi);
        const __nv_bfloat16 mid = __float2bfloat16(r1);
        out[idx] = plane == 0 ? hi : (plane == 1 ? mid : __float2bfloat16(r1 - __bfloat162float(mid)));
    }
}
cudaError_t launch_prepack_weight(const float* w, __nv_bfloat16* out, int Cout, int Cin_total, int taps, int nseg,
                                  const int* segc, int shuffle, int planes, cudaStream_t st, const float* gamma) {
    prepack_weight_kernel<<<1024, 256, 0, st>>>(w, out, Cout, Cin_total, taps, nseg, segc[0], nseg > 1 ? segc[1] : 0,
                                                nseg > 2 ? segc[2] : 0, shuffle, planes, gamma);
    return cudaGetLastError();
}

// LayerNorm folded into a linear layer (GemmParams::ln_stats_in): bias' = bias + W beta (fp32 W), and
// wsum_c = sum_k W'[c, k] taken over the bf16-ROUNDED packed weights, so that mean * wsum cancels exactly what the
// tensor core accumulated for a constant row.  One warp per output channel.
__global__ void fold_ln_kernel(const float* __restrict__ w, const float* __restrict__ beta, const float* __restrict__ bias,
                               const __nv_bfloat16* __restrict__ packed, int Kp, int Cout, int Cin, float* __restrict__ bias_out,
                               float* __restrict__ wsum) {
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (c >= Cout) return;
    float b = 0.f, s = 0.f;
    for (int k = lane; k < Cin; k += 32) b = fmaf(w[(size_t)c * Cin + k], beta[k], b);
    for (int k = lane; k < Kp; k += 32) s += __bfloat162float(packed[(size_t)c * Kp + k]);
    b = warp_sum(b);
    s = warp_sum(s);
    if (lane == 0) { bias_out[c] = bias[c] + b; wsum[c] = s; }
}
cudaError_t launch_fold_ln(const float* w, const float* beta, const float* bias, const __nv_bfloat16* packed, int Kp, int Cout, int Cin,
                           float* bias_out, float* wsum, cudaStream_t st) {
    fold_ln_kernel<<<(Cout * 32 + 255) / 256, 256, 0, st>>>(w, beta, bias, packed, Kp, Cout, Cin, bias_out, wsum);
    return cudaGetLastError();
}

__global__ void permute_bias_shuffle_kernel(const float* __restrict__ b, float* __restrict__ out, int Cout) {
    const int ro = blockIdx.x * blockDim.x + threadIdx.x;
    if (ro >= Cout) return;
    const int cq = Cout >> 2;
    const int q = ro / cq, c = ro - q * cq;
    out[ro] = b[c * 4 + q];
}
// Block-diagonal weight of TWO 3x3 conv layers that read different inputs, as ONE layer over the concatenated input
// (GemmParams::gc_on): out [2 half, 2 Cin, 3, 3] fp32 (+ bias [2 half]); output rows are interleaved in 32-row chunks -
// chunk b = [layer A rows 16 b .. 16 b + 15 | layer B rows 16 b .. 16 b + 15] - so one 32-column accumulator chunk holds both
// layers' outputs of the same 16 channels.  Layer A sees input channels [0, Cin), layer B [Cin, 2 Cin); the rest is zero, and
// a zero product adds exactly 0 to the fp32 accumulator: the fused GEMM is bit-identical to the two separate ones.
__global__ void build_blockdiag2_kernel(const float* __restrict__ wa, const float* __restrict__ wb, const float* __restrict__ ba,
                                        const float* __restrict__ bb, float* __restrict__ w_out, float* __restrict__ b_out, int half,
                                        int Cin, int taps) {
    const long long per_row = (long long)2 * Cin * taps;
    const long long total = (long long)2 * half * per_row;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int ro = (int)(idx / per_row);
        const long long rem = idx - (long long)ro * per_row;
        const int c = (int)(rem / taps), tap = (int)(rem - (long long)c * taps);
        const int blk = ro >> 5, within = ro & 31, net = within >> 4, ch = blk * 16 + (within & 15);
        float v = 0.f;
        if (net == 0 && c < Cin) v = wa[((size_t)ch * Cin + c) * taps + tap];
        else if (net == 1 && c >= Cin) v = wb[((size_t)ch * Cin + (c - Cin)) * taps + tap];
        w_out[idx] = v;
        if (rem == 0) b_out[ro] = net == 0 ? ba[ch] : bb[ch];
    }
}
cudaError_t launch_build_blockdiag2(const float* wa, const float* wb, const float* ba, const float* bb, float* w_out, float* b_out,
                                    int half, int Cin, int taps, cudaStream_t st) {
    if (half % 16 != 0) return cudaErrorInvalidValue;
    build_blockdiag2_kernel<<<256, 256, 0, st>>>(wa, wb, ba, bb, w_out, b_out, half, Cin, taps);
    return cudaGetLastError();
}

cudaError_t launch_permute_bias_shuffle(const float* b, float* out, int Cout, cudaStream_t st) {
    permute_bias_shuffle_kernel<<<(Cout + 255) / 256, 256, 0, st>>>(b, out, Cout);
    return cudaGetLastError();
}

// Factorized-prior table: softplus(matrix), bias, tanh(factor), median (see bottleneck_kernel).
__global__ void eb_table_kernel(const float* m0, const float* b0, const float* f0, const float* m1, const float* b1,
                                const float* f1, const float* m2, const float* b2, const float* f2, const float* m3,
                                const float* b3, const float* f3, const float* m4, const float* b4,
                                const float* quantiles, float* tab, int Cz) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Cz) return;
    float* t = tab + c;                                   // parameter-major: entry k of channel c at tab[k * Cz + c]
    auto softplus = [](float x) { return x > 20.f ? x : log1pf(expf(x)); };   // F.softplus(beta=1, threshold=20)
    for (int i = 0; i < 3; ++i) {
        t[i * Cz] = softplus(m0[c * 3 + i]);
        t[(3 + i) * Cz] = b0[c * 3 + i];
        t[(6 + i) * Cz] = tanhf(f0[c * 3 + i]);
    }
    const float* mm[3] = {m1, m2, m3};
    const float* bb[3] = {b1, b2, b3};
    const float* ff[3] = {f1, f2, f3};
    for (int l = 0; l < 3; ++l) {
        float* tt = t + (9 + 15 * l) * Cz;
        for (int i = 0; i < 9; ++i) tt[i * Cz] = softplus(mm[l][c * 9 + i]);
        for (int i = 0; i < 3; ++i) {
            tt[(9 + i) * Cz] = bb[l][c * 3 + i];
            tt[(12 + i) * Cz] = tanhf(ff[l][c * 3 + i]);
        }
    }
    float* tl = t + 54 * Cz;
    for (int i = 0; i < 3; ++i) tl[i * Cz] = softplus(m4[c * 3 + i]);
    tl[3 * Cz] = b4[c];
    t[58 * Cz] = 0.f; t[59 * Cz] = 0.f;
    t[60 * Cz] = quantiles[c * 3 + 1];
    t[61 * Cz] = 0.f; t[62 * Cz] = 0.f; t[63 * Cz] = 0.f;
}
cudaError_t launch_eb_table(const float* const* ptrs, float* tab, int Cz, cudaStream_t st) {
    eb_table_kernel<<<(Cz + 127) / 128, 128, 0, st>>>(ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5], ptrs[6],
                                                      ptrs[7], ptrs[8], ptrs[9], ptrs[10], ptrs[11], ptrs[12],
                                                      ptrs[13], ptrs[14], tab, Cz);
    return cudaGetLastError();
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ a, __nv_bfloat16* __restrict__ o, long long n, long long lo_off) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        store_bf16_planes(o + i, lo_off, a[i]);
}
cudaError_t launch_f32_to_bf16(const float* a, __nv_bfloat16* o, long long n, long long lo_off, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    f32_to_bf16_kernel<<<512, 256, 0, st>>>(a, o, n, lo_off);
    return cudaGetLastError();
}

// strided form: `cols` consecutive columns of every row (row pitch `ld` in both tensors)
__global__ void f32_to_bf16_cols_kernel(const float* __restrict__ a, __nv_bfloat16* __restrict__ o, long long rows, int cols, int ld,
                                        long long lo_off) {
    const long long total = rows * cols;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / cols;
        const int c = (int)(i - r * cols);
        store_bf16_planes(o + r * ld + c, lo_off, a[r * ld + c]);
    }
}
cudaError_t launch_f32_to_bf16_cols(const float* a, __nv_bfloat16* o, long long rows, int cols, int ld, long long lo_off, cudaStream_t st) {
    if (rows == 0) return cudaSuccess;
    f32_to_bf16_cols_kernel<<<256, 256, 0, st>>>(a, o, rows, cols, ld, lo_off);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// Synthesis (tmae_synthesize: recon.synthesize on the engine).  The per-call pointers come from the IoBlock.
// ---------------------------------------------------------------------------------------------------------
// io->syn_y_hat (f32 [rows, Cy], the caller's channels-last y_hat) -> bf16, the A operand of g_s.0.  n4 = elements / 4.
__global__ void __launch_bounds__(256)
synth_input_kernel(__nv_bfloat16* __restrict__ out, long long n4, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    const float4* a = reinterpret_cast<const float4*>(io->syn_y_hat);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = a[i];
        uint2 pk;
        pk.x = pack_bf16x2(v.x, v.y);
        pk.y = pack_bf16x2(v.z, v.w);
        reinterpret_cast<uint2*>(out)[i] = pk;
    }
}

cudaError_t launch_synth_input(__nv_bfloat16* out, long long n, cudaStream_t st, const IoBlock* io) {
    if (n % 4 != 0) return cudaErrorInvalidValue;
    const long long n4 = n / 4;
    const unsigned blocks = (unsigned)((n4 + 255) / 256 < 1184 ? (n4 + 255) / 256 : 1184);
    TMAE_CARVEOUT_ONCE(synth_input_kernel);
    return launch_k(synth_input_kernel, dim3(blocks > 0 ? blocks : 1), dim3(256), 0, st, true, out, n4, io);
}

// MAE decoder input (recon.forward_decoder, MCM.py:636-665, with its quirk reproduced): decoder_embed's output emb f32
// [N*K, D] -> residual stream x f32 [N*T, D], T = L + 1.  Row 0 of an image is its token 0; row t >= 1 takes
// j = ids_restore[t - 1], clamped to [0, L) so that no id can read out of bounds: token j + 1 if j < K - 1, else mask_token.
// Every row then adds decoder_pos_embed[t].  Also writes the bf16 copy of x and one (sum, sum of squares) partial per row and
// 32-column chunk - the statistics block 0's LayerNorm-folded QKV reads, in the layout the proj / fc2 store phases write.
// Thread = 4 columns of one row, 8 threads = one chunk.
__global__ void __launch_bounds__(256)
synth_unshuffle_kernel(const float* __restrict__ emb, const float* __restrict__ mask_token, const float* __restrict__ pos,
                       float* __restrict__ x, __nv_bfloat16* __restrict__ x_bf, float* __restrict__ stats, int N, int K, int L, int D,
                       const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    const int T = L + 1, q = D / 4;
    const long long total = (long long)N * T * q;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = i < total;                       // every lane takes part in the chunk reduction below
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    long long row = 0;
    int c = 0;
    if (ok) {
        row = i / q;
        c = (int)(i - row * q) * 4;
        const int n = (int)(row / T), t = (int)(row - (long long)n * T);
        const float* src = emb + (size_t)n * K * D;
        if (t > 0) {
            long long j = io->syn_ids[(size_t)n * L + (t - 1)];
            j = j < 0 ? 0 : (j >= L ? L - 1 : j);
            src = j < K - 1 ? emb + ((size_t)n * K + (size_t)j + 1) * D : mask_token;
        }
        const float4 a = *reinterpret_cast<const float4*>(src + c);
        const float4 p = __ldg(reinterpret_cast<const float4*>(pos + (size_t)t * D + c));
        v = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
        *reinterpret_cast<float4*>(x + (size_t)row * D + c) = v;
        uint2 pk;
        pk.x = pack_bf16x2(v.x, v.y);
        pk.y = pack_bf16x2(v.z, v.w);
        *reinterpret_cast<uint2*>(x_bf + (size_t)row * D + c) = pk;
    }
    float s1 = (v.x + v.y) + (v.z + v.w);
    float s2 = fmaf(v.x, v.x, v.y * v.y) + fmaf(v.z, v.z, v.w * v.w);
#pragma unroll
    for (int sh = 1; sh < 8; sh <<= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, sh);
        s2 += __shfl_xor_sync(0xffffffffu, s2, sh);
    }
    if (ok && (threadIdx.x & 7) == 0) reinterpret_cast<float2*>(stats)[row * (D / 32) + c / 32] = make_float2(s1, s2);
}

cudaError_t launch_synth_unshuffle(const float* emb, const float* mask_token, const float* pos, float* x, __nv_bfloat16* x_bf, float* stats,
                                   int N, int K, int L, int D, cudaStream_t st, const IoBlock* io) {
    if (D % 32 != 0 || K < 1 || K > L) return cudaErrorInvalidValue;
    const long long total = (long long)N * (L + 1) * (D / 4);
    TMAE_CARVEOUT_ONCE(synth_unshuffle_kernel);
    return launch_k(synth_unshuffle_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, true, emb, mask_token, pos, x, x_bf,
                    stats, N, K, L, D, io);
}

// decoder_pred's output preds bf16 [N*T, P*P*3] -> io->syn_x_hat f32 [N, 3, S, S] (recon.unpatchify, MCM.py:524-546: (p, q, c)
// order within a patch); row 0 of every image is dropped.  Thread = 4 consecutive pixels of one row of one channel.
__global__ void __launch_bounds__(256)
synth_unpatchify_kernel(const __nv_bfloat16* __restrict__ preds, int N, int P, int gw, const IoBlock* __restrict__ io) {
    pdl_wait();
    pdl_launch_dependents();
    float* __restrict__ xh = io->syn_x_hat;
    const int S = gw * P, S4 = S / 4, T = gw * gw + 1, ld = P * P * 3;
    const long long total = (long long)N * 3 * S * S4;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int X = (int)(i % S4) * 4;
        long long r = i / S4;
        const int y = (int)(r % S);
        r /= S;
        const int ch = (int)(r % 3), n = (int)(r / 3);
        const int hh = y / P, p = y - hh * P, ww = X / P, qq = X - ww * P;
        const __nv_bfloat16* src = preds + ((size_t)n * T + 1 + hh * gw + ww) * ld + (p * P + qq) * 3 + ch;
        const float4 o = make_float4(__bfloat162float(src[0]), __bfloat162float(src[3]), __bfloat162float(src[6]), __bfloat162float(src[9]));
        *reinterpret_cast<float4*>(xh + (((size_t)n * 3 + ch) * S + y) * S + X) = o;
    }
}

cudaError_t launch_synth_unpatchify(const __nv_bfloat16* preds, int N, int P, int gw, cudaStream_t st, const IoBlock* io) {
    if (P % 4 != 0) return cudaErrorInvalidValue;
    const long long total = (long long)N * 3 * gw * P * gw * P / 4;
    const long long want = (total + 255) / 256;
    TMAE_CARVEOUT_ONCE(synth_unpatchify_kernel);
    return launch_k(synth_unpatchify_kernel, dim3((unsigned)(want < 2368 ? want : 2368)), dim3(256), 0, st, true, preds, N, P, gw, io);
}

}  // namespace tmae
