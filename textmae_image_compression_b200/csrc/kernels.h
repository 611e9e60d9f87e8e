// Host-side launch prototypes of every kernel in the library (internal; the public ABI is include/tmae.h).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tmae.h"
#include "gemm.cuh"

namespace tmae {

// Per-call pointers of one forward, resident in device memory: kernels captured in a CUDA graph read the caller's
// buffers through it, so one instantiated graph serves every call of that batch size.
struct IoBlock {
    const float* imgs;
    const float* scores;
    tmae_outputs out;
    const int32_t* z_symbols;        // decode: z symbols [N, Cz, s/4, s/4] (range-coder order)
    const int32_t* y_symbols;        // decode: y symbols [N, Cy * s * s], per image slice by slice in (c, y, x) order
    const uint8_t* y_data;           // decode from streams (tmae_decompress_streams): image n's y stream is bytes
    const int64_t* y_offsets;        //   [y_offsets[n], y_ends[n]) of y_data; likewise z.  Streams packed back to back:
    const int64_t* y_ends;           //   y_ends = y_offsets + 1; inside image containers: the ranges image_parse_kernel wrote
    const uint8_t* z_data;
    const int64_t* z_offsets;
    const int64_t* z_ends;
    int32_t* status;                 //   [N] per-image coder status (RANS_ST_* bits, and IMG_ST_* from the container parse)
    const uint8_t* img_data;         // decode from image containers (tmae_decompress_images): container n is bytes
    const int64_t* img_offsets;      //   [img_offsets[n], img_ends[n]) of img_data, inside [0, img_n_bytes).  Containers packed back
    const int64_t* img_ends;         //   to back: img_ends = img_offsets + 1; the tiles of pictures: the ranges picture_parse_kernel wrote
    long long img_n_bytes;
    int64_t* img_ids_restore;        //   [N, L] out: the canonical ids_restore of every container
    int64_t* img_ids_keep;           //   [N, K] out (may be null): the kept patch ids of every container
    const int64_t* pic_offsets;      // decode from picture containers (tmae_decompress_pictures): picture p is bytes
                                     //   [pic_offsets[p], pic_offsets[p + 1]) of img_data; its T tiles are images p T .. p T + T - 1
    int64_t* pic_ranges;             //   [2 N] out: begin, then end byte of every tile container (-> img_offsets / img_ends)
    int32_t* pic_status;             //   [P] out: PIC_ST_HEADER, ORed with the status of every tile of the picture
    int pic_P, pic_H, pic_W;         //   pictures and their height / width
    const float* syn_y_hat;          // synthesis (tmae_synthesize): y_hat f32 [N, s, s, Cy] in,
    const int64_t* syn_ids;          //   ids_restore [N, L] in,
    float* syn_x_hat;                //   x_hat f32 [N, 3, S, S] out
};

// gemm_tc.cu
cudaError_t gemm_tc_configure();
const GemmOptions& gemm_options();
bool conv_geom(int s, int n_img, ConvGeom* g);
// Host-only and pure: the launch a GEMM step of shape `s` runs.  false = no launch form fits (a forced form the shape rules out).
bool gemm_resolve(const GemmShape& s, GemmLaunch* out);
cudaError_t gemm_launch(const GemmLaunch& L, const GemmParams* d_params, const GemmParams* d_next, int next_groups, cudaStream_t stream);

// mask.cu
cudaError_t launch_mask_select(const float* scores, int N, int L, int K, int softmax_isa, int64_t* ids_shuffle,
                               int64_t* ids_restore, int64_t* ids_keep, cudaStream_t st, const IoBlock* io = nullptr);

// attention.cu
cudaError_t attention_configure(int T);
cudaError_t launch_attention(const __nv_bfloat16* qkv, __nv_bfloat16* out, int N, int T, int H, int C, float scale,
                             cudaStream_t st);
// tcgen05 / TMEM attention (T <= 192): Q / K / V by TMA out of the qkv matrix, S and O in tensor memory
bool attention_tc_supported(int T);   // kernel limits (Tp <= 384: shared memory and the 512 TMEM columns)
bool attention_tc_eligible(int T);    // policy: the tcgen05 kernel whenever it is supported (TMAE_NO_TC_ATTN=1 -> mma.sync kernel)
int attention_tc_tp(int T);
// mode: 1 = full form, 2 = several streams share the GPU (lite form for short rows), 3 = duo (two heads per tile, T = 65; opt-in)
bool attention_tc_describe(int T, int H, int N, int mode, int* out12);        // host-only: the plan for (T, H, N) in `mode`
void attention_tc_boxes(int T, int H, int mode, int* q_rows, int* kv_rows);   // TMA box rows of the Q map and of the K / V map
cudaError_t launch_attention_tc(const CUtensorMap* map_q, const CUtensorMap* map_kv, const __nv_bfloat16* qkv, __nv_bfloat16* out, int N,
                                int T, int H, int C, float scale, cudaStream_t st, long long* dbg = nullptr, int mode = 1);
// head dim 32 (the MAE decoder of the synthesis plan): the mma.sync kernel above with 32-column heads, qkv columns [3][H][32]
bool attention_hd32_supported(int T);     // K and V of all T keys fit shared memory (T <= ~1300)
cudaError_t launch_attention_hd32(const __nv_bfloat16* qkv, __nv_bfloat16* out, int N, int T, int H, float scale, cudaStream_t st);
// precise mode: fp32 softmax attention on CUDA cores over split-bf16 (hi + lo plane) q, k, v; writes both planes
cudaError_t launch_attention_f32(const __nv_bfloat16* qkv, long long qkv_lo, __nv_bfloat16* out, long long out_lo, int N,
                                 int T, int H, int C, float scale, cudaStream_t st);

// elementwise.cu
cudaError_t launch_gather_patches(const float* imgs, const int64_t* ids_keep, __nv_bfloat16* patches, float* x,
                                  const float* cls_token, const float* pos_embed, int N, int S, int grid_w, int K,
                                  int T, int C, int in_chans, int patch, long long lo_off, cudaStream_t st,
                                  const IoBlock* io = nullptr);
cudaError_t launch_layernorm(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out, float* out_f32,
                             int rows, int C, int T, int drop_cls, float eps, long long lo_off, cudaStream_t st,
                             const IoBlock* io = nullptr);
cudaError_t launch_bottleneck(const float* z, const float* eb_tab, long long rows, int Cz, float* lik, int32_t* sym,
                              float* zhat, __nv_bfloat16* zhat_bf, long long lo_off, int s4, double* rate_acc, int rows_per_image,
                              int16_t* sym16,
                              cudaStream_t st, const IoBlock* io = nullptr);
cudaError_t launch_gaussian_slice(const float* y, const float* mu, const float* sigma, long long rows, int ld, int col0,
                                  int cs, float* lik, int32_t* sym, float* yhat, __nv_bfloat16* yhat_bf, long long lo_off,
                                  int ld_bf, int s, double* rate_acc, const float* scale_table, int n_table, int16_t* sym16,
                                  int32_t* idx, cudaStream_t st, const IoBlock* io = nullptr);
// decode side (the range coder's symbols back to the latents)
cudaError_t launch_z_dequantize(const float* eb_tab, long long rows, int Cz, int hw, __nv_bfloat16* zhat_bf, long long lo_off,
                                cudaStream_t st, const IoBlock* io);
cudaError_t launch_slice_indexes(const float* sigma, long long rows, int ld, int col0, int cs, int hw, const float* scale_table,
                                 int n_table, cudaStream_t st, const IoBlock* io);
cudaError_t launch_slice_dequantize(const float* mu, long long rows, int ld, int col0, int cs, int hw, float* yhat,
                                    __nv_bfloat16* yhat_bf, long long lo_off, cudaStream_t st, const IoBlock* io);
cudaError_t launch_pack_nchw_i32(const int32_t* src, int32_t* dst, int N, int hw, int C, cudaStream_t st);
cudaError_t launch_gaussian_flat(const float* y, const float* mu, const float* sigma, long long n, float* lik,
                                 int32_t* sym, float* yhat, cudaStream_t st);
cudaError_t launch_rate_finalize(const double* rate_acc, int N, double pixels_per_image, float* bpp,
                                 double* rate_sums, cudaStream_t st, const IoBlock* io = nullptr);
// copies the workspace-resident results the caller asked for (io->out.{y,z,mu,sigma,y_hat,ids_keep})
cudaError_t launch_copy_outputs(const IoBlock* io, const float* y, const float* z, const float* mu, const float* sigma,
                                const float* yhat, const int64_t* ids_keep, long long n_y, long long n_z, long long n_ids,
                                cudaStream_t st);
cudaError_t launch_prepack_weight(const float* w, __nv_bfloat16* out, int Cout, int Cin_total, int taps, int nseg,
                                  const int* segc, int shuffle, int planes, cudaStream_t st, const float* gamma = nullptr);
cudaError_t launch_fold_ln(const float* w, const float* beta, const float* bias, const __nv_bfloat16* packed, int Kp, int Cout, int Cin,
                           float* bias_out, float* wsum, cudaStream_t st);
cudaError_t launch_build_blockdiag2(const float* wa, const float* wb, const float* ba, const float* bb, float* w_out, float* b_out,
                                    int half, int Cin, int taps, cudaStream_t st);
cudaError_t launch_permute_bias_shuffle(const float* b, float* out, int Cout, cudaStream_t st);
cudaError_t launch_eb_table(const float* const* ptrs, float* tab, int Cz, cudaStream_t st);
// synthesis (tmae_synthesize): y_hat in, the MAE decoder's input rows, x_hat out (per-call pointers from the IoBlock)
cudaError_t launch_synth_input(__nv_bfloat16* out, long long n, cudaStream_t st, const IoBlock* io);
cudaError_t launch_synth_unshuffle(const float* emb, const float* mask_token, const float* pos, float* x, __nv_bfloat16* x_bf, float* stats,
                                   int N, int K, int L, int D, cudaStream_t st, const IoBlock* io);
cudaError_t launch_synth_unpatchify(const __nv_bfloat16* preds, int N, int P, int gw, cudaStream_t st, const IoBlock* io);
cudaError_t launch_f32_to_bf16(const float* a, __nv_bfloat16* o, long long n, long long lo_off, cudaStream_t st);
cudaError_t launch_f32_to_bf16_cols(const float* a, __nv_bfloat16* o, long long rows, int cols, int ld, long long lo_off, cudaStream_t st);

// rans.cu: the entropy coder (compressai's rANS format)
enum : int32_t {                     // per-stream status bits (include/tmae.h TMAE_RANS_*)
    RANS_ST_OVERRUN = 1,             // decode read past the end of the stream (those words read as 0)
    RANS_ST_UNFINISHED = 2,          // decode ended with a state other than the encoder's initial one, or words left over
    RANS_ST_BAD_INDEX = 4,           // an index outside the table set (coded with table 0)
    RANS_ST_RANGE = 8,               // encode: a symbol whose escape value does not fit 31 bits (coded as 0)
    RANS_ST_OVERFLOW = 16,           // encode: the packed output does not fit the capacity (stream not written)
    RANS_ST_MALFORMED = 32,          // decode: byte range negative / not a multiple of 4, or an escape longer than 8 nibbles
};
struct CdfTables {                   // one quantised-CDF table set on the device (tmae_set_cdf_tables)
    int n = 0;                       // tables
    int entries = 0;                 // sum of the cdf lengths
    int* cdf = nullptr;              // [entries] the cdfs back to back, then meta
    int* meta = nullptr;             // [3 * n]: start in cdf, cdf length, offset of every table
    uint4* enc = nullptr;            // [entries]: symbol v of table t at start + v: {start | freq << 16, reciprocal shift, reciprocal lo, hi}
};
struct RansDecState {                // decoder state of one stream (laned format: one lane) between the stages of a decode plan
    unsigned long long x;
    unsigned pos, pad;               // next word; laned format: pad = the lane's end word
};
struct RansDecArgs {
    const int* cdf = nullptr;        // CdfTables::cdf (meta follows the entries)
    int entries = 0, n_tab = 0;
    int lanes = 0;                   // 0: compressai's format (warp per stream); 1..32: laned format (thread per lane), state [s * lanes + l]
    int use_smem = 0, streams_per_block = 1;                 // set by launch_rans_decode
    const uint8_t* data = nullptr;   // streams: bytes [begins[s], ends[s]) of data (packed back to back: ends = begins + 1)
    const int64_t* begins = nullptr;
    const int64_t* ends = nullptr;
    const int32_t* indexes = nullptr;                        // [s * idx_stride + i]; nullptr: table (i / idx_div)
    long long idx_stride = 0;
    int idx_div = 1;
    int32_t* symbols = nullptr;      // [s * sym_stride + i]
    long long sym_stride = 0;
    int n_streams = 0, begin = 0, end = 0;                   // symbols [begin, end) of every stream
    int init = 1, fin = 1;           // init: read the two head words; fin: check the final state
    int status_reset = 1;            // init: overwrite status[s] (else OR into it)
    RansDecState* state = nullptr;   // between stages (init == 0 reads it, fin == 0 writes it)
    int32_t* status = nullptr;
    const IoBlock* io = nullptr;     // non-null: data / begins / ends / status (and, io_stream 1, the indexes io->out.y_indexes)
    int io_stream = 0;               //   come from the IoBlock: 1 = the y streams, 2 = the z streams
};
int pmf_to_quantized_cdf(const float* pmf, int n, int32_t* cdf_out);          // host; cdf_out holds n + 1 entries
long long rans_bound_bytes(long long n);
int rans_build_tables(const int32_t* cdf, int n, int stride, const int32_t* len, const int32_t* off, CdfTables* out,
                      char* err, size_t err_len);                            // host arrays in; uploads (synchronous)
void rans_free_tables(CdfTables* t);
long long rans_bound_lanes_bytes(long long n, int lanes);                    // laned format; -1 for n < 0 or lanes outside 1..32
// lanes = 0: compressai's format; 1..32: the laned format (scratch: n_streams * lanes regions of cap_words)
cudaError_t launch_rans_encode(const int32_t* sym, const int32_t* idx, int n_streams, int n_per, int lanes, const CdfTables& tab,
                               uint2* rec, uint32_t* scratch, long long cap_words, long long* n_words, uint8_t* out, long long capacity,
                               int64_t* offsets, int32_t* status, cudaStream_t st);
cudaError_t launch_rans_decode(RansDecArgs a, cudaStream_t st);

// container.cu: image containers (DESIGN.md section 7)
enum : int32_t {                     // per-image status bits of the container parse (include/tmae.h TMAE_IMG_*)
    IMG_ST_HEADER = 64,              // magic / version / reserved bits, or section lengths other than the container's byte range
    IMG_ST_CONFIG = 128,             // geometry, accuracy mode or lane counts other than the handle's / call's
    IMG_ST_MODEL = 256,              // model tag other than the handle's
    IMG_ST_IDS = 512,                // a patch id >= L, or two equal ids
};
constexpr uint32_t kImageMagic = 0x45414D54u;    // bytes "TMAE"
struct ImageFields {                 // what the handle writes into (and expects of) words 1 to 4 of a container
    uint32_t word1;                  // version | accuracy mode << 8 | W_y << 16 | W_z << 24
    uint32_t word2;                  // img_size | patch_size << 16
    uint32_t word3;                  // K
    uint32_t tag;                    // model tag
    int L, K, id_bits;               // patches, kept patches, bits per packed id
};
// Images packed as the tiles of pictures (tmae_compress_pictures): every group of T consecutive images is one picture, whose
// header and length table take the 4 (4 + T) bytes in front of its first tile.  T = 0: plain image containers, back to back.
struct PictureGroup {
    int T = 0;                       // tiles per picture
    uint32_t hw = 0;                 // word 2 of the picture header: H | W << 16
    int64_t* offsets = nullptr;      // [N / T + 1] out: picture offsets
    int32_t* status = nullptr;       // [N / T] out: OR of the picture's tile status
};
// after the encodes of N images (stream offsets / status of each kind): container n at offsets[n] of out
cudaError_t launch_image_pack(const int64_t* ids_keep, const uint8_t* y_bytes, const int64_t* y_off, const int32_t* y_st,
                              const uint8_t* z_bytes, const int64_t* z_off, const int32_t* z_st, const ImageFields& f, int N,
                              uint8_t* out, long long capacity, int64_t* offsets, int32_t* status, cudaStream_t st,
                              const PictureGroup& g = PictureGroup());
// the containers of io->img_*: canonical ids_restore (io->img_ids_restore), io->img_ids_keep when non-null, io->status, and the
// stream ranges [4 N] (z begin, z end, y begin, y end)
cudaError_t launch_image_parse(const IoBlock* io, const ImageFields& f, int N, int64_t* ranges, cudaStream_t st);

// picture.cu: pictures of any size as tiles of img_size (DESIGN.md section 7, "The picture container")
constexpr int32_t PIC_ST_HEADER = 1024;          // include/tmae.h TMAE_PIC_HEADER
constexpr uint32_t kPictureMagic = 0x50414D54u;  // bytes "TMAP"
// pictures f32 [P, 3, H, W] -> tiles f32 [P T, 3, S, S] and grey tiles u8 [P T, S, S] (either may be null), zero-padded; the grey
// tiles are cut from gray u8 [P, H, W], or made from the RGB (cv2 RGB2GRAY of the 8-bit pixels) when gray is null
cudaError_t launch_picture_tile(const float* imgs, const uint8_t* gray, int P, int H, int W, int S, float* tiles,
                                uint8_t* gray_tiles, cudaStream_t st);
// tiles f32 [P T, 3, S, S] -> canvas f32 [P, 3, H, W]
cudaError_t launch_picture_untile(const float* tiles, int P, int H, int W, int S, float* canvas, cudaStream_t st);
// the picture headers of io->pic_*: io->pic_ranges, io->pic_status (S = img_size)
cudaError_t launch_picture_parse(const IoBlock* io, int P, int S, cudaStream_t st);
// io->pic_status[p] |= io->status of its T tiles
cudaError_t launch_picture_status(const IoBlock* io, int P, int T, cudaStream_t st);

// ---- patch-score generation (scores.cu; generate_scores_file.py:19-31, utils/map.py, utils/distribution.py) ----
constexpr int kScoreMaxLevels = 16;
struct ScoreGeom {
    int H, W, S;                           // grey image, side of the resized maps (224)
    int levels;                            // quadtree levels whose nodes may split (min(h, w) > 5); deeper nodes are leaves
    int flag_total;                        // split-decision flags per image = sum of 4^d over those levels
    int large_levels, large_nodes, large_cta_total, small_nodes;
    int h[kScoreMaxLevels + 1], w[kScoreMaxLevels + 1];       // node size per level: int(h / 2) of the level above
    int flag_off[kScoreMaxLevels + 1];
    int chunks[kScoreMaxLevels], large_node_off[kScoreMaxLevels], large_ctas[kScoreMaxLevels];
    double scale_x_crop, scale_y_crop, scale_x_full, scale_y_full;   // cv2.resize source/destination ratios
};
bool score_geometry(int H, int W, int S, ScoreGeom* out);
size_t score_workspace_bytes(const ScoreGeom& g, int n);
cudaError_t launch_generate_scores(const uint8_t* gray, int n, const ScoreGeom& g, float* scores, uint8_t* s_map, uint8_t* t_map,
                                   uint8_t* seg_out, void* workspace, cudaStream_t st);

}  // namespace tmae
