// Parameter block of the multi-tap / multi-segment GEMM engine (linear layers, 1x1 convs and 3x3 convs as
// 9 row-shifted GEMM taps over a zero-haloed channels-last activation matrix).  One GemmParams lives in device
// memory per layer (per group member for grouped launches); the kernels index it with blockIdx.z.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace tmae {

constexpr int kBlockM = 128;      // UMMA M (cta_group::1)
constexpr int kBlockK = 64;       // 64 bf16 = 128 B = one 128B-swizzle atom row
constexpr int kMaxSegs = 18;      // 3 concatenated channel segments x up to 6 split-bf16 terms (precise layers)
constexpr int kMaxTaps = 9;

// Row spaces.  Every activation matrix is COMPACT channels-last: pixel (n, y, x) of an s x s grid is row n*s*s + y*s + x.
//   IN_LINEAR  plain GEMM rows (tokens)
//   IN_COMPACT plain GEMM rows that are pixels of an s x s grid (g_a, patch embed): only the token remap needs (n, j)
//   IN_CONV    3x3 convolution: the A tile of a CTA is a 4-D TMA box [64 ch, s (x), box_n images, box_y rows] of the
//              compact tensor (accumulator row r = (yl * box_n + nl) * s + x); a tap (dy, dx) shifts the box
//              coordinates and TMA zero-fills what falls outside the image, so there is no halo / im2col buffer and no
//              wasted rows when s*box_y*box_n == 128.  conv_reuse: ONE box with a row of halo above and below
//              ([64, s, box_n, box_y + 2]) is loaded per (channel block, dx) and serves the three dy taps through
//              shared-memory descriptor offsets of box_n*s rows (a multiple of the 8-row swizzle atom).
//
// Precise layers (split-bf16, TMAE_FLAG_PRECISE_*): every operand is a pair of bf16 planes (hi = bf16(v),
// lo = bf16(v - hi)) and a product a*w is issued as three tensor-core terms a_hi*w_hi + a_lo*w_hi + a_hi*w_lo
// (relative error ~2^-17 instead of 2^-9; the dropped a_lo*w_lo term is ~2^-18).  The terms are simply MORE K SEGMENTS
// of the same main loop: segment list (A_hi, W_hi), (A_lo, W_hi), (A_hi, W_lo) per concatenated source, the weights hold
// the hi planes of a tap followed by its lo planes (seg_b_kb0 points each segment at its weight columns).
// TMAE_FLAG_PRECISE_X6 carries fp32 exactly: three planes (hi, mid, lo = 24 mantissa bits) and the six terms
// hi*hi + mid*hi + hi*mid + mid*mid + lo*hi + hi*lo (dropped terms ~2^-24).
enum InMode : int { IN_LINEAR = 0, IN_COMPACT = 1, IN_CONV = 2 };
enum RowMap : int {
    MAP_SAME = 0,        // out row = the pixel's / token's own compact row
    MAP_TO_TOKEN,        // compact (n, j) -> token row n*T + 1 + j
    MAP_S2,              // stride-2 subsample -> compact grid of side s/2
    MAP_SHUF,            // PixelShuffle(2): column quadrant q -> compact grid of side 2s
    MAP_GATHER1          // row = gather_ids[m] + 1 (pos-embed lookup)
};
enum Act : int { ACT_NONE = 0, ACT_GELU = 1, ACT_HALF_TANH = 2 };
enum OutType : int { OUT_NONE = 0, OUT_BF16 = 1, OUT_F32 = 2 };

struct OutSpec {
    void* ptr;
    int ld;        // elements per row
    int dtype;     // OutType
    int map;       // RowMap
    long long lo_off;   // bf16 outputs feeding a precise layer: plane layout, see store_bf16x4_planes (0 one plane, > 0 two planes
                        // that many elements apart, < 0 three planes -lo_off apart)
};

struct alignas(64) GemmParams {
    CUtensorMap a_map[kMaxSegs];      // linear: [rows, C_seg] box 64 x 128; conv: (C_seg, x, n, y) box 64 x s x box_n x box_y (+2 rows if conv_reuse)
    CUtensorMap b_map;                // [N, Kpacked] bf16, box 64 x block_n, SWIZZLE_128B
    CUtensorMap b_map_pair;           // pair (cta_group::2) launches: box 64 x block_n / 2 (each CTA of the pair stages half of B)
    CUtensorMap out_map;              // TMA-store epilogue only: out[0] as [rows, N] bf16, box 32 x 128 (conv: (N, x, n, y), box 32 x s x box_n x box_y), SWIZZLE_64B
    // raw views of the same operands (CUDA-core checker kernel)
    const __nv_bfloat16* a_ptr[kMaxSegs];
    int a_ld[kMaxSegs];
    int a_cols[kMaxSegs];             // valid channels of the segment
    long long a_rows[kMaxSegs];       // valid rows of the segment's matrix
    const __nv_bfloat16* b_ptr;
    int b_ld;                         // Kpacked
    // K loop
    int num_segs;
    int seg_kblocks[kMaxSegs];        // ceil(C_seg / 64)
    int seg_b_kb0[kMaxSegs];          // first k-block of the segment's weights inside one tap of the packed B matrix
    int b_kb_per_tap;                 // k-blocks per tap of the packed B matrix (precise layers: hi planes then lo planes)
    int num_taps;                     // 1, or 9 for IN_CONV: taps in (kh, kw) row-major order, shift (kw - 1, kh - 1)
    // problem
    int M;                            // linear: rows; conv: m_tiles * 128 (virtual rows of the tile grid)
    int N;                            // output channels
    int block_n;
    // input row space geometry
    int in_mode;
    int s;                            // side of the pixel grid
    int K;                            // s*s
    int T;                            // tokens per image (K + 1)
    int n_img;                        // conv: images
    int box_y, box_n;                 // conv: image rows / images per CTA tile
    int rows_used;                    // conv: s * box_y * box_n (<= 128) accumulator rows that hold pixels
    int y_tiles;                      // conv: ceil(s / box_y)
    int pair_ok;                      // b_map_pair is valid (linear layer, block_n % 32 == 0)
    int tma_store_ok;                 // out_map is valid (linear: the tile is 128 consecutive output rows; conv: the 4-D box of the tile)
    int conv_reuse;                   // conv: one haloed A box per (channel block, dx) serves the three dy taps
    int a_halo_rows;                  // conv_reuse: (box_y + 2) * box_n * s rows of 128 B per A box
    // epilogue
    const float* bias;                // [N] (already permuted for MAP_SHUF)
    int act;
    const float* resid;               // optional fp32 addend, read at row map `resid_map`
    int resid_ld;
    int resid_map;
    const int64_t* gather_ids;        // MAP_GATHER1
    OutSpec out[2];
    // LayerNorm folded into the GEMMs around it (bf16 mode, encoder blocks).  Consumer (QKV / fc1): A = bf16(x) of the raw
    // residual stream, the weights carry gamma (W' = W diag(gamma), bias' = bias + W beta) and the epilogue applies
    //     out = rstd_r * (acc - mean_r * wsum_c) + bias'_c,   wsum_c = sum_k W'[c, k] (of the bf16-rounded W'),
    // with (sum x, sum x^2) of row r summed from ln_stats_in.  Producer (proj / fc2, fp32 residual epilogue): writes one
    // (sum v, sum v^2) partial per output row and 32-column chunk to ln_stats_out (plain stores, a fixed slot per chunk:
    // deterministic and independent of tiling / batch size) and bf16(v) to xbf_out.
    const float* ln_stats_in;         // [rows][ln_chunks][2] or nullptr
    const float* ln_wsum;             // [N]
    float ln_inv_c, ln_eps;
    int ln_chunks;                    // C / 32 of the normalised rows
    float* ln_stats_out;              // [rows][N / 32][2] or nullptr
    __nv_bfloat16* xbf_out;           // [rows][N] or nullptr
    // Gaussian conditional fused into the LAST layer of cc_transform_mean[i] and cc_transform_scale[i] (MCM.py:761-776): the two
    // 3x3 convs (80 -> 32 channels, different inputs) run as ONE block-diagonal GEMM with 64 output columns - [0, 32) = mu,
    // [32, 64) = sigma of slice i - and the epilogue (thread = pixel) quantises y, evaluates the likelihoods, emits symbols /
    // scale-table indexes / y_hat and adds the pixel's log2-likelihood to its image's rate.  No gaussian_slice_kernel launch, mu
    // and sigma never travel through HBM to be read back.
    int gc_on;                        // 1 = encoder (EPI_GAUSS), 2 = decoder: mu, sigma and indexes only (EPI_GAUSS_IDX)
    int gc_col0;                      // first channel of the slice in the [rows, gc_ld] tensors
    int gc_ld;                        // Cy
    int gc_pixels;                    // pixels per image (rate accumulator index = row / gc_pixels)
    const float* gc_y;                // [rows, Cy] latent
    float* gc_mu;                     // [rows, Cy] workspace copies (parity outputs)
    float* gc_sigma;
    float* gc_yhat;                   // [rows, Cy] fp32 y_hat before LRP (the LRP net's last layer adds to it)
    __nv_bfloat16* gc_yhat_bf;        // [rows, Cy] bf16 copy (+ planes, gc_yhat_lo): support of the later slices
    long long gc_yhat_lo;
    double* gc_rate;                  // [images] sum of log2 likelihoods
    const float* gc_table;            // scale table for y_indexes (may be null)
    int gc_ntable;
    const void* gc_io;                // IoBlock*: the caller's y_likelihoods / y_symbols / y_symbols_i16 / y_indexes of this call
    double flops;                     // flops of this GEMM as the reference would count them for the rows computed (profiling)
    int mma_terms;                    // tensor-core products issued per algorithmic product: 1, or 3 / 6 for precise (split-bf16) layers
    long long* dbg_ticks;             // optional [ctas][8] globaltimer stamps of the kernel phases (bring-up)
};

}  // namespace tmae
