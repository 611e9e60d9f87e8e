/* tmae.h - C ABI of the B200-native TextMAE compression forward path (libtmae_b200.so).
 *
 * Drop-in boundary for ONE path of tmkhang1999/TextMAE-Image-Compression: everything
 * `MCM.forward(imgs, total_scores)` computes up to the rate
 * (reference models/Compression/MCM.py:590-634 forward_encoder, :714-787 rate half of forward,
 *  models/Compression/loss/rd_loss.py:15-20 bpp).  The reference has no FFI of its own (it is pure
 * Python); these entry points are what a ctypes / pybind binding of that path binds
 * (INTEGRATION.md shows the reference-side stub).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary.
 *   - every pointer is a DEVICE pointer unless the name starts with h_ (tmae_forward_host).
 *   - activations are channels-last: a reference tensor [N, C, h, w] is passed as [N, h, w, C]
 *     (the Python host returns .permute(0,3,1,2) views so callers see the reference shape).
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no host
 *     synchronisation and no allocation once the workspace for that batch size exists.
 *   - return value: 0 on success, otherwise a tmae_status; tmae_last_error() gives the text.
 *     Nothing throws or aborts across the ABI.  There is no CPU fallback.
 */
#ifndef TMAE_H_
#define TMAE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TMAE_ABI_VERSION 3
#if defined(__GNUC__)
#define TMAE_API __attribute__((visibility("default")))
#else
#define TMAE_API
#endif

typedef enum {
    TMAE_OK = 0,
    TMAE_EINVAL = 1,      /* bad argument / geometry the reference rejects (K > L, K not (4j)^2, size mismatch) */
    TMAE_ECUDA = 2,       /* CUDA runtime / driver error; text in tmae_last_error */
    TMAE_ESTATE = 3,      /* call order (weights missing / not finalized) */
    TMAE_ENOMEM = 4
} tmae_status;

typedef enum { TMAE_F32 = 0, TMAE_BF16 = 1, TMAE_F16 = 2 } tmae_dtype;

/* Constructor arguments of the reference module, MCM.__init__ (MCM.py:34-52), hot-path subset. */
typedef struct {
    int32_t img_size;            /* 224 */
    int32_t patch_size;          /* 16  */
    int32_t in_chans;            /* 3   */
    int32_t encoder_embed_dim;   /* 768 */
    int32_t encoder_depth;       /* 12  */
    int32_t encoder_num_heads;   /* 12  */
    int32_t decoder_embed_dim;   /* 512 : fixes the g_a channel ladder (MCM.py:77-93) */
    float   mlp_ratio;           /* 4.0 */
    int32_t latent_depth;        /* 384 */
    int32_t hyperprior_depth;    /* 192 */
    int32_t num_slices;          /* 12  */
    int32_t num_keep_patches;    /* 144 */
    float   ln_eps;              /* 1e-6 */
    int32_t softmax_isa;         /* 16 / 8: ATen CPU softmax lane order mirrored by the mask kernel (0 = 16) */
    int32_t flags;               /* TMAE_FLAG_* */
} tmae_config;

#define TMAE_FLAG_SKIP_DEAD_LRP 1u   /* rate-only: skip lrp_transform[6..11] (their y_hat feeds only g_s) */
#define TMAE_FLAG_DEBUG_SIMT    2u   /* bring-up only: run GEMM/conv layers on the CUDA-core checker kernel */
#define TMAE_FLAG_SHARE_SM      4u   /* several handles/streams run concurrently on this GPU: size every launch so that
                                        CTAs of two kernels can share an SM (<= half the shared memory each) */
/* Accuracy modes ("precise"): the named layers run with split-bf16 operands - every activation and weight is a pair of
 * bf16 planes (hi, lo) and each product is three tensor-core terms a_hi*w_hi + a_lo*w_hi + a_hi*w_lo accumulated in fp32
 * (relative product error ~2^-17 instead of 2^-9), so that the quantised symbols round(y - mu) match the reference's fp32
 * arithmetic up to rounding-boundary ties (north_star; MCM.py:735, 761-783). */
#define TMAE_FLAG_PRECISE_RATE  8u   /* g_a, h_a, h_s_*, cc_transform_*, lrp_transform: everything after the encoder */
#define TMAE_FLAG_PRECISE_ALL   16u  /* the encoder as well (patch embed, Block linears, fp32 softmax attention) */
#define TMAE_FLAG_PRECISE_X6    32u  /* with either of the above: three bf16 planes per operand (24 mantissa bits = fp32
                                        carried exactly) and six terms per product - fp32-equivalent arithmetic */

/* Outputs of one forward; any pointer may be NULL (that output is skipped).
 * N = batch, L = (img/patch)^2, K = num_keep_patches, s = sqrt(K), Cy = latent_depth, Cz = hyperprior_depth. */
typedef struct {
    float*   y_likelihoods;   /* [N, s, s, Cy]      == out["likelihoods"]["y"] (MCM.py:787,801), NHWC */
    float*   z_likelihoods;   /* [N, s/4, s/4, Cz]  == out["likelihoods"]["z"] (MCM.py:741,801), NHWC */
    int32_t* y_symbols;       /* [N, s, s, Cy]      round(y - mu)       (MCM.py:776)  */
    int32_t* z_symbols;       /* [N, s/4, s/4, Cz]  round(z - median)   (MCM.py:742-744) */
    float*   y_hat;           /* [N, s, s, Cy]      after LRP           (MCM.py:783-786) */
    float*   z_hat;           /* [N, s/4, s/4, Cz] */
    float*   y;               /* [N, s, s, Cy]      g_a output          (MCM.py:735) */
    float*   z;               /* [N, s/4, s/4, Cz]  h_a output          (MCM.py:739) */
    float*   mu;              /* [N, s, s, Cy]      per-slice means     (MCM.py:762-763) */
    float*   sigma;           /* [N, s, s, Cy]      per-slice raw scales(MCM.py:767-768) */
    float*   x_remain;        /* [N, K, C]          encoder output      (MCM.py:631-632) */
    float*   bpp;             /* [N]                per-image rate, rd_loss.py:15-20 with N = 1 */
    double*  rate_sums;       /* [2]                {sum log2 likelihood over the batch, N * S * S pixels} */
    int64_t* ids_shuffle;     /* [N, L]             MCM.get_ids_shuffle return value (MCM.py:423) */
    int64_t* ids_restore;     /* [N, L]             argsort(ids_shuffle) (MCM.py:580) */
    int64_t* ids_keep;        /* [N, K]             ids_shuffle[:, :K]   (MCM.py:583) */
    int16_t* y_symbols_i16;   /* [N, s, s, Cy]      y_symbols saturated to int16 (compact form for the host / the coder) */
    int16_t* z_symbols_i16;   /* [N, s/4, s/4, Cz]  z_symbols saturated to int16 */
    int32_t* y_indexes;       /* [N, s, s, Cy]      GaussianConditional.build_indexes(sigma): scale-table bucket of every
                                                    element (MCM.py:839; needs tmae_set_scale_table) */
} tmae_outputs;

/* HOST destinations of tmae_forward_host (pinned memory for full speed); any pointer may be NULL.  This is what the
 * reference's forward hands back to its caller - likelihoods (MCM.py:801) - plus the symbols and the per-image rate. */
typedef struct {
    float*   bpp;             /* [N] */
    double*  rate_sums;       /* [2] */
    float*   y_likelihoods;   /* [N, s, s, Cy] */
    float*   z_likelihoods;   /* [N, s/4, s/4, Cz] */
    int16_t* y_symbols;       /* [N, s, s, Cy] */
    int16_t* z_symbols;       /* [N, s/4, s/4, Cz] */
    int64_t* ids_restore;     /* [N, L] (the reference returns it on the CPU, MCM.py:580) */
} tmae_host_outputs;

typedef struct tmae_handle tmae_handle;

/* Lifetime -------------------------------------------------------------------------------------- */
TMAE_API int  tmae_abi_version(void);
/* Validates geometry exactly like the reference would fail (see tmae_status) and creates a handle on the
 * current CUDA device. */
TMAE_API int  tmae_create(const tmae_config* cfg, tmae_handle** out);
TMAE_API void tmae_destroy(tmae_handle* h);
TMAE_API const char* tmae_last_error(const tmae_handle* h);   /* h may be NULL: error of the last failed tmae_create */

/* Weights: one call per state-dict entry, names exactly as in MCM.state_dict() (SURVEY 8b), e.g.
 * "encoder_blocks.3.attn.qkv.weight".  `data` may be a device or host pointer (cudaMemcpyDefault); the library
 * copies it, so the caller may free it on return.  Unknown names (buffers; the decoder side - g_s, decoder_*,
 * mask_token - unless tmae_enable_synthesis was called) are ignored and reported through *ignored when non-NULL. */
TMAE_API int  tmae_set_weight(tmae_handle* h, const char* name, const void* data, int dtype, int ndim,
                     const int64_t* shape, int* ignored);
/* Checks that every tensor the path needs is present, prepacks to bf16 tensor-core layouts, precomputes
 * softplus/tanh of the factorized-prior parameters.  Synchronises the device. */
TMAE_API int  tmae_finalize_weights(tmae_handle* h);

/* Synthesis: x_hat from y_hat on the engine (g_s, the MAE decoder and unpatchify; the reference's MCM.py:789-792).
 * tmae_enable_synthesis, before tmae_finalize_weights (after it, it marks the weights unfinalized as tmae_set_weight does),
 * makes tmae_set_weight accept the decoder-side tensors (g_s.*, decoder_embed.*, mask_token, decoder_pos_embed,
 * decoder_blocks.*, decoder_norm.*, decoder_pred.*) and tmae_finalize_weights require them (TMAE_ESTATE naming a missing one;
 * TMAE_EINVAL for a wrong shape: g_s.{0,2,4,6}.weight are ConvTranspose2d [cin, cout, 1, 1], mask_token [1, 1, Dd],
 * decoder_pos_embed [1, L + 1, Dd]).  TMAE_EINVAL for depth < 1, a head count that does not divide decoder_embed_dim, a
 * head dim other than 32, or a TMAE_FLAG_DEBUG_SIMT handle (or TMAE_NO_TMA_STORE set).  Synthesis runs bf16 operands with fp32 accumulation, residual
 * stream, LayerNorm statistics and softmax in every accuracy mode (the TMAE_FLAG_PRECISE_* flags govern the rate path). */
TMAE_API int  tmae_enable_synthesis(tmae_handle* h, int decoder_depth, int decoder_num_heads);
/* x_hat f32 [N, 3, S, S] (NCHW) from y_hat f32 [N, s, s, Cy] (channels-last, as the forward and the decodes write it) and
 * ids_restore i64 [N, L]: recon.synthesize computed on the engine.  y_hat and x_hat 16-byte aligned.  Asynchronous: no host
 * synchronisation and, once the plan of this N exists, no allocation; replays as one CUDA graph per N.  An ids_restore value
 * outside [0, L) is clamped (never read out of bounds); the pixels are then unspecified.  TMAE_ESTATE unless synthesis is
 * enabled and the weights are finalized. */
TMAE_API int  tmae_synthesize(tmae_handle* h, const float* y_hat, const int64_t* ids_restore, int N, float* x_hat, void* stream);

/* Scale table of the reference's GaussianConditional (testing.py:223 model.update(force=True) builds it with
 * compressai's get_scale_table(): 64 log-spaced scales 0.11..256): enables out->y_indexes.  Host or device pointer,
 * ascending, n <= 256. */
TMAE_API int  tmae_set_scale_table(tmae_handle* h, const float* table, int n);

/* Workspace: grown on demand inside tmae_forward; this makes the growth explicit (e.g. before CUDA-graph capture). */
TMAE_API size_t tmae_workspace_bytes(const tmae_handle* h, int N);
TMAE_API int  tmae_reserve(tmae_handle* h, int N);

/* The hot path --------------------------------------------------------------------------------- */
/* imgs: f32 [N, in_chans, S, S] NCHW contiguous; scores: f32 [N, L].  (MCM.forward arguments, MCM.py:714) */
TMAE_API int  tmae_forward(tmae_handle* h, const float* imgs, const float* scores, int N,
                  const tmae_outputs* out, void* stream);
/* Same call with HOST buffers: h_imgs / h_scores (pinned for full speed) are copied in on `stream`, the
 * forward runs, and every non-NULL member of `hout` (likelihoods, int16 symbols, ids_restore, per-image bpp) is
 * copied back on the same stream; `out` (device pointers, optional) as in tmae_forward. */
TMAE_API int  tmae_forward_host(tmae_handle* h, const float* h_imgs, const float* h_scores, int N,
                       const tmae_host_outputs* hout, const tmae_outputs* out, void* stream);
/* Teacher-forced entry for parity tests: run the rate half only (MCM.py:739-787) from a given latent
 * y f32 [N, s, s, Cy]. */
TMAE_API int  tmae_forward_from_latent(tmae_handle* h, const float* y, int N, const tmae_outputs* out, void* stream);
/* Slice-wise teacher forcing for parity tests: as above, but every slice reads the GIVEN y_hat f32 [N, s, s, Cy] (the
 * reference's) as the support of the slices before it (MCM.py:756-761, 780) instead of this run's own, so one
 * rounding-boundary flip cannot cascade through mu of the later slices. */
TMAE_API int  tmae_forward_from_latent_forced(tmae_handle* h, const float* y, const float* y_hat_support, int N,
                                     const tmae_outputs* out, void* stream);
/* Encoder only (MCM.forward_encoder, MCM.py:590-634): fills out->x_remain / ids_*. */
TMAE_API int  tmae_forward_encoder(tmae_handle* h, const float* imgs, const float* scores, int N,
                          const tmae_outputs* out, void* stream);

/* Decode (MCM.decompress, MCM.py:896-968, with the range decoder left to the caller) ---------------------------- *
 * The rate half of the forward with y replaced by the caller's symbols: z_hat -> h_s -> per slice group mu / sigma ->
 * scale-table indexes -> (caller decodes the group's symbols) -> y_hat = symbols + mu -> lrp_transform.  The range decoder
 * needs a group's indexes before it can produce that group's symbols, so the decode runs in stages: tmae_decode_begin,
 * then tmae_decode_step for every slice group in order.  Symbols go in and indexes come out in the range coder's order
 * (per image, slice by slice, each (c, y, x): the layout of the lists the reference passes to encode_with_indexes /
 * decode_stream, i.e. NCHW of [Cy, s, s]); z_hat / y_hat / mu / sigma come out channels-last like every other output.
 * A handle decodes what a handle of the same configuration (flags included) encoded, bit for bit: the same layers run
 * with the same launch shapes.  Any other call on the handle between begin and the last step, or a step out of order, ends
 * the decode (that step and the next return TMAE_ESTATE). */
/* Host-only: the slice groups of the decode (first slice, slice count each); returns their count (7 for 12 slices), or
 * -TMAE_EINVAL.  first_slice / n_slices may be NULL (count only), else they hold `capacity` entries. */
TMAE_API int  tmae_decode_groups(int num_slices, int* first_slice, int* n_slices, int capacity);
/* z_symbols: i32 [N, Cz, s/4, s/4].  Writes out->z_hat (if non-NULL) and the indexes of group 0 into out->y_indexes
 * (required, i32 [N, Cy*s*s]).  Needs the scale table (tmae_set_scale_table; TMAE_ESTATE without it). */
TMAE_API int  tmae_decode_begin(tmae_handle* h, const int32_t* z_symbols, int N, const tmae_outputs* out, void* stream);
/* y_symbols: i32 [N, Cy*s*s] in coder order, of which the region of `group` is read.  Dequantises the group, runs its
 * lrp_transform and writes the indexes of group + 1 into out->y_indexes; after the last group out->y_hat (and out->mu /
 * out->sigma when non-NULL) are complete.  Other members of `out` are ignored. */
TMAE_API int  tmae_decode_step(tmae_handle* h, int group, const int32_t* y_symbols, const tmae_outputs* out, void* stream);

/* Entropy coder: compressai 1.2.4's rANS bitstream (BufferedRansEncoder / RansDecoder *_with_indexes over rans64, precision 16,
 * 4-bit bypass escapes; DESIGN.md section 7) on the GPU.  A stream is a sequence of 32-bit words, stored little-endian; its
 * byte length is a multiple of 4 and at least 8.  Streams of a batch are packed back to back: stream i is bytes
 * [offsets[i], offsets[i + 1]) of `data` (device memory, 4-byte aligned).  Per-stream status: 0 = the stream decoded to its
 * end exactly (final state equals the encoder's initial state, every word consumed), otherwise TMAE_RANS_* bits.  Input
 * bytes may be anything: every read is bounded by the stream's length (past the end reads as 0 and sets a bit). */
#define TMAE_MODEL_GAUSSIAN     0    /* GaussianConditional: one table per scale-table entry, index = build_indexes(sigma) */
#define TMAE_MODEL_BOTTLENECK   1    /* EntropyBottleneck: one table per channel, index = channel */
#define TMAE_RANS_OVERRUN       1    /* decode read past the end of the stream */
#define TMAE_RANS_UNFINISHED    2    /* decode ended in another state than the encoder started from, or left words unread */
#define TMAE_RANS_BAD_INDEX     4    /* an index outside the table set (coded / decoded with table 0) */
#define TMAE_RANS_RANGE         8    /* encode: a symbol too far outside its table (escape value >= 2^31; coded as 0) */
#define TMAE_RANS_OVERFLOW      16   /* encode: the packed streams exceed `capacity` (this stream was not written) */
#define TMAE_RANS_MALFORMED     32   /* decode: bad byte range, or an escape longer than 8 nibbles */
/* Host-only: compressai's pmf_to_quantized_cdf at precision 16.  h_pmf [n] -> h_cdf [n + 1] (0 .. 65536, strictly
 * increasing).  TMAE_EINVAL for a negative / non-finite / all-zero pmf. */
TMAE_API int  tmae_pmf_to_quantized_cdf(const float* h_pmf, int n, int32_t* h_cdf);
/* Host-only: bytes that always suffice for one stream of n symbols (10 words per symbol + 2), -1 for n < 0. */
TMAE_API int64_t tmae_rans_bound(int64_t n_symbols);
/* Installs one table set: cdf [n_tables, stride] in compressai's padded _quantized_cdf layout, cdf_lengths / offsets [n_tables]
 * (_cdf_length / _offset); host or device pointers, copied.  Every table must have length >= 3, start at 0, increase strictly
 * and end at 65536 (TMAE_EINVAL otherwise).  Bottleneck: n_tables must equal hyperprior_depth. */
TMAE_API int  tmae_set_cdf_tables(tmae_handle* h, int model, const int32_t* cdf, int n_tables, int stride,
                                  const int32_t* cdf_lengths, const int32_t* offsets);
/* encode_with_indexes + flush of n_streams streams of n_per_stream symbols each (symbols / indexes i32 [n_streams, n_per_stream]):
 * packed into out (capacity bytes; n_streams * tmae_rans_bound(n_per_stream) always suffices), offsets i64 [n_streams + 1],
 * status i32 [n_streams].  Scratch memory is the handle's, grown on the first call of a larger size. */
TMAE_API int  tmae_rans_encode(tmae_handle* h, int model, const int32_t* symbols, const int32_t* indexes, int n_streams,
                               int n_per_stream, uint8_t* out, int64_t capacity, int64_t* offsets, int32_t* status, void* stream);
/* decode_with_indexes of n_streams streams: indexes / symbols i32 [n_streams, n_per_stream], status i32 [n_streams]. */
TMAE_API int  tmae_rans_decode(tmae_handle* h, int model, const uint8_t* data, const int64_t* offsets, int n_streams,
                               const int32_t* indexes, int n_per_stream, int32_t* symbols, int32_t* status, void* stream);
/* The whole decode from bitstreams, enqueued without a host synchronisation: per image one y stream (every slice in order, the
 * symbols in the order of tmae_decode_step) and one z stream (z symbols in NCHW order, table = channel).  The z streams are
 * decoded with the bottleneck tables, then each slice group's y symbols with the Gaussian tables and the indexes the decode has
 * just computed.  Writes out->z_hat / y_hat and, when non-NULL, out->mu / sigma / y_indexes (other members ignored); status
 * i32 [N].  Needs the scale table and both table sets, the Gaussian set with one table per scale-table entry (TMAE_ESTATE). */
TMAE_API int  tmae_decompress_streams(tmae_handle* h, const uint8_t* y_data, const int64_t* y_offsets, const uint8_t* z_data,
                                      const int64_t* z_offsets, int N, const tmae_outputs* out, int32_t* status, void* stream);

/* Laned rANS format (DESIGN.md section 7): a stream of n symbols with W lanes (1 <= W <= 32) is, as little-endian 32-bit words,
 * {W, len[0..W), lane 0 .. lane W-1}: lane l holds the compressai stream (as above) of the symbols l, l + W, l + 2W, ... with their
 * indexes, len[l] its byte length (a multiple of 4, at least 8; a lane without symbols is the 8 flush bytes).  The stream is
 * 4 (1 + W) + sum len bytes.  The lanes decode in parallel (one thread each), so a stream's decode chain is W times shorter.
 * Decode status per stream: TMAE_RANS_MALFORMED for a header with another W or lengths that do not add up; every read is
 * bounded by its own lane (TMAE_RANS_OVERRUN); every lane must end in the encoder's initial state with all its words read
 * (TMAE_RANS_UNFINISHED); the stream's status is the OR over its lanes.  The calls below take lanes in 1..32 and reject it, and
 * null pointers, with TMAE_EINVAL (a null handle included); without the needed tables they return TMAE_ESTATE. */
/* Host-only: bytes that always suffice for one laned stream of n symbols (4 (1 + W) + 4 (10 n + 2 W)); -1 for n < 0 or W outside
 * 1..32. */
TMAE_API int64_t tmae_rans_bound_lanes(int64_t n_symbols, int lanes);
/* tmae_rans_encode in the laned format: n_streams * tmae_rans_bound_lanes(n_per_stream, lanes) bytes of `out` always suffice. */
TMAE_API int  tmae_rans_encode_lanes(tmae_handle* h, int model, const int32_t* symbols, const int32_t* indexes, int n_streams,
                                     int n_per_stream, int lanes, uint8_t* out, int64_t capacity, int64_t* offsets, int32_t* status,
                                     void* stream);
/* tmae_rans_decode of laned streams. */
TMAE_API int  tmae_rans_decode_lanes(tmae_handle* h, int model, const uint8_t* data, const int64_t* offsets, int n_streams,
                                     const int32_t* indexes, int n_per_stream, int lanes, int32_t* symbols, int32_t* status, void* stream);
/* tmae_decompress_streams of laned streams: y streams of y_lanes lanes (lanes assigned on the symbol's position in the image's
 * whole y stream, so a lane's state carries across the slice groups), z streams of z_lanes lanes.  Replays as one CUDA graph per
 * (N, y_lanes, z_lanes). */
TMAE_API int  tmae_decompress_streams_lanes(tmae_handle* h, const uint8_t* y_data, const int64_t* y_offsets, int y_lanes,
                                            const uint8_t* z_data, const int64_t* z_offsets, int z_lanes, int N,
                                            const tmae_outputs* out, int32_t* status, void* stream);

/* Image containers (DESIGN.md section 7): one self-contained byte string per image - a 28-byte header (magic "TMAE", version,
 * accuracy mode, lane counts, img_size, patch_size, K, model tag, z and y stream lengths), the kept patch ids ids_keep[0..K)
 * bit-packed in max(1, bit_length(L - 1)) bits each, then the z and the y stream exactly as tmae_rans_encode(_lanes) writes them.
 * Lanes: 0 = compressai's format, 1..32 = the laned format with that many lanes.  Status bits above the coder's (ORed with them
 * per image): */
#define TMAE_IMG_HEADER         64   /* decode: bad magic / version / reserved bits, or section lengths that do not add up to the
                                        container's byte range (or a range outside [0, n_bytes)) */
#define TMAE_IMG_CONFIG         128  /* decode: img_size, patch_size, K, accuracy mode or lane counts other than the handle's / call's */
#define TMAE_IMG_MODEL          256  /* decode: model tag other than the handle's (other scale table or CDF tables) */
#define TMAE_IMG_IDS            512  /* decode: a patch id >= L, or two equal ids */
/* Host-only: FNV-1a (32-bit) over the scale table (fp32) and then, Gaussian set first, every table's cdf length, offset and cdf
 * entries (int32), all little-endian: what a container's model tag must equal.  TMAE_ESTATE until the scale table and both CDF
 * table sets are installed; TMAE_EINVAL for null pointers.  The synthesis weights are not covered. */
TMAE_API int  tmae_model_tag(const tmae_handle* h, uint32_t* tag);
/* Host-only: bytes that always suffice for the containers of N images (the ABI's worst case of both streams plus the header and
 * the patch ids, per image); -1 for a null handle, N < 1 or lanes outside {0} and 1..32. */
TMAE_API int64_t tmae_images_bound(const tmae_handle* h, int N, int y_lanes, int z_lanes);
/* The forward of N images (imgs / scores as tmae_forward), then both rANS encodes and the packing of one container per image,
 * all enqueued on `stream` without a host synchronisation.  Container n is bytes [offsets[n], offsets[n + 1]) of `out` (device,
 * 4-byte aligned; capacity bytes, tmae_images_bound always suffices); offsets i64 [N + 1] (8-byte aligned), status i32 [N]
 * (device, 4-byte aligned): the coder's
 * encode bits, TMAE_RANS_OVERFLOW when the container does not fit `capacity` (not written).  Needs the scale table and both CDF
 * table sets (TMAE_ESTATE). */
TMAE_API int  tmae_compress_images(tmae_handle* h, const float* imgs, const float* scores, int N, int y_lanes, int z_lanes,
                                   uint8_t* out, int64_t capacity, int64_t* offsets, int32_t* status, void* stream);
/* Decode of N containers, bytes [offsets[n], offsets[n + 1]) of data (device, 4-byte aligned, n_bytes long; offsets i64 [N + 1]
 * on the device; offsets, ids_restore and out->ids_keep 8-byte aligned, status 4-byte aligned: TMAE_EINVAL otherwise), enqueued without a host synchronisation: a parse-and-validate kernel, then the decode of
 * tmae_decompress_streams(_lanes) from the streams inside the containers, then (x_hat non-NULL) the synthesis of
 * tmae_synthesize.  Writes out->y_hat / z_hat (and out->ids_keep i64 [N, K] when non-NULL), ids_restore i64 [N, L] - the
 * canonical one: ids_restore[ids_keep[j]] = j, the other positions in ascending order K .. L-1 - and x_hat f32 [N, 3, S, S].
 * status i32 [N]: 0 = decoded exactly; TMAE_IMG_* for a container the parse refuses (its streams are then not read), TMAE_RANS_*
 * for streams that do not decode.  A bad container never affects another.  y_lanes / z_lanes: the lane counts every container
 * must carry.  Replays as one CUDA graph per (N, y_lanes, z_lanes); x_hat needs tmae_enable_synthesis (TMAE_ESTATE). */
TMAE_API int  tmae_decompress_images(tmae_handle* h, const uint8_t* data, int64_t n_bytes, const int64_t* offsets, int N,
                                     int y_lanes, int z_lanes, const tmae_outputs* out, int64_t* ids_restore, float* x_hat,
                                     int32_t* status, void* stream);

/* Picture containers (DESIGN.md section 7, "The picture container"): a picture of any size H x W (1..65535 each) in one byte
 * string.  The picture is zero-padded on the bottom / right to whole tiles of side S = img_size and cut into T = rows * cols tiles
 * in raster order (tiling.py's policy); every tile is coded as the image container tmae_compress_images writes for it, with the
 * scores the score generator makes from the tile's grey pixels (out_side = img_size).  Little-endian 32-bit words: magic "TMAP",
 * version 1 (byte 0; bytes 1-3 reserved, 0), H | W << 16, T, the byte length of each tile container, then the T tile containers.
 * A picture is 4 (4 + T) + sum of the lengths bytes.  Status bit above the image containers' (ORed with its tiles' status): */
#define TMAE_PIC_HEADER         1024 /* decode: bad magic / version / reserved bits, H / W / T other than the call's, lengths that are
                                        not multiples of 4 or do not add up to the picture's byte range (or a range outside
                                        [0, n_bytes)); every tile of the picture is then refused as well (TMAE_IMG_HEADER) */
/* Stand-alone: pictures f32 [P, 3, H, W] -> tiles f32 [P T, 3, tile, tile] and grey tiles u8 [P T, tile, tile] (either output may
 * be NULL), zero padding, equal to tiling.tile_image.  The grey tiles are cut from gray u8 [P, H, W], or, with gray NULL, made from
 * the RGB as OpenCV's cvtColor(RGB2GRAY) of v = saturate_u8(rint(255 x)): (9798 R + 19235 G + 3735 B + 16384) >> 15. */
TMAE_API int  tmae_picture_tiles(const float* imgs, const uint8_t* gray, int P, int H, int W, int tile, float* tiles,
                                 uint8_t* gray_tiles, void* stream);
/* Stand-alone: tiles f32 [P T, 3, tile, tile] -> canvas f32 [P, 3, H, W], padding dropped (tiling.untile_image of each picture). */
TMAE_API int  tmae_picture_untile(const float* tiles, int P, int H, int W, int tile, float* canvas, void* stream);
/* Host-only: H, W and T of the picture in h_data [n_bytes] and the lane counts of its first tile (any output may be NULL).
 * TMAE_EINVAL for bytes that are not a picture (magic, version, reserved bits, a first tile that is not an image container, or a
 * T other than the tile grid of H x W at the first tile's img_size). */
TMAE_API int  tmae_picture_geometry(const uint8_t* h_data, int64_t n_bytes, int* H, int* W, int* T, int* y_lanes, int* z_lanes);
/* Host-only: bytes that always suffice for P pictures of H x W; -1 for a null handle, P < 1, H or W outside 1..65535 or lanes
 * outside {0} and 1..32. */
TMAE_API int64_t tmae_pictures_bound(const tmae_handle* h, int P, int H, int W, int y_lanes, int z_lanes);
/* P pictures imgs f32 [P, 3, H, W] (gray u8 [P, H, W] or NULL as in tmae_picture_tiles) to one picture container each, enqueued on
 * `stream` without a host synchronisation: the tiling, the score generator on the grey tiles, the forward of the P T tiles, both
 * rANS encodes and the pack, which writes the tile containers straight into the picture layout.  Picture p is bytes
 * [offsets[p], offsets[p + 1]) of `out` (capacity bytes; tmae_pictures_bound always suffices).  status i32 [P]: the OR of its tiles'
 * encode bits, or TMAE_RANS_OVERFLOW.  P T <= 65535.  Argument checks as tmae_compress_images (out and status 4-byte aligned,
 * offsets 8-byte aligned), and in_chans must be 3.  Scratch (tiles, grey tiles, scores) is the handle's, grown on first use. */
TMAE_API int  tmae_compress_pictures(tmae_handle* h, const float* imgs, const uint8_t* gray, int P, int H, int W, int y_lanes,
                                     int z_lanes, uint8_t* out, int64_t capacity, int64_t* offsets, int32_t* status, void* stream);
/* Decode of P pictures of H x W, bytes [offsets[p], offsets[p + 1]) of data (n_bytes long), enqueued without a host
 * synchronisation: the picture parse, then the image-container decode of the P T tiles (tmae_decompress_images), replayed as one
 * CUDA graph per (tiles, lanes, H x W); then, x_hat non-NULL, the synthesis of the tiles and their untiling into x_hat
 * f32 [P, 3, H, W].  tile_out (may be NULL): y_hat / z_hat / ids_keep and the other decode outputs of the tiles, as in
 * tmae_decompress_images; ids_restore i64 [P T, L] (may be NULL).  status i32 [P]: TMAE_PIC_HEADER ORed with the status of every
 * tile of the picture.  A bad picture never affects another; the pixels of a picture with nonzero status are unspecified, but every
 * write stays inside its canvas.  Alignment: data and status 4 bytes, offsets, ids_restore and ids_keep 8, y_hat and x_hat 16. */
TMAE_API int  tmae_decompress_pictures(tmae_handle* h, const uint8_t* data, int64_t n_bytes, const int64_t* offsets, int P, int H,
                                       int W, int y_lanes, int z_lanes, const tmae_outputs* tile_out, int64_t* ids_restore,
                                       float* x_hat, int32_t* status, void* stream);

/* Stand-alone operators on the path (each mirrors one reference call) ---------------------------------- */
/* MCM.get_ids_shuffle + random_masking index work (MCM.py:364-423, 579-583). Outputs may be NULL. */
TMAE_API int  tmae_mask_select(const float* scores, int N, int L, int K, int softmax_isa,
                      int64_t* ids_shuffle, int64_t* ids_restore, int64_t* ids_keep, void* stream);
/* GaussianConditional eval forward + quantize_ste (MCM.py:771-776) on n elements. */
TMAE_API int  tmae_gaussian_rate(const float* y, const float* mu, const float* sigma, int64_t n,
                        float* likelihood, int32_t* symbols, float* y_hat, void* stream);
/* EntropyBottleneck eval forward + quantize_ste (MCM.py:741-744): z f32 [rows, Cz] channels-last. */
TMAE_API int  tmae_bottleneck_rate(tmae_handle* h, const float* z, int64_t rows,
                          float* likelihood, int32_t* symbols, float* z_hat, void* stream);

/* [N, hw, C] channels-last int32 -> [N, C, hw]: the order the reference feeds its range coder, slice by slice in
 * (c, y, x) order (MCM.py:867-873), for symbols and indexes alike. */
TMAE_API int  tmae_pack_nchw_i32(const int32_t* nhwc, int32_t* nchw, int N, int hw, int C, void* stream);

/* Patch-score generation (the reference's offline generator, generate_scores_file.py:19-31 = utils/map.py:6-60
 * Division_Merge_Segmented + laplacian, utils/distribution.py:5-16 cal_patch_score, min-max normalisation): what
 * `total_scores` of MCM.forward is made of.  gray: uint8 [n, height, width] (cv2.imread(..., IMREAD_GRAYSCALE) of each
 * image, all of one size); out_side = 224 in the reference (any multiple of 16).  Any output may be NULL.  Bit-exact
 * with the reference's numpy / OpenCV arithmetic (integer and float64 work; see csrc/scores.cu). */
typedef struct {
    float*   scores;          /* [n, (out_side/16)^2]  fp32, NaN where an image's scores are all equal (0/0, like numpy) */
    uint8_t* s_map;           /* [n, out_side, out_side]  Division_Merge_Segmented(img, (out_side, out_side)) */
    uint8_t* t_map;           /* [n, out_side, out_side]  laplacian(img, (out_side, out_side)) of the segmented image */
    uint8_t* segmented;       /* [n, height, width]       the image after Recursion / Merge (utils/map.py:35-42) */
} tmae_score_outputs;
TMAE_API size_t tmae_scores_workspace_bytes(int n, int height, int width, int out_side);   /* 0 = invalid geometry */
/* workspace: device memory, 256-byte aligned, >= tmae_scores_workspace_bytes(...); n <= 65535 images per call. */
TMAE_API int  tmae_generate_scores(const uint8_t* gray, int n, int height, int width, int out_side,
                          const tmae_score_outputs* out, void* workspace, size_t workspace_bytes, void* stream);

/* Side-information coder of the reference's eval CLI: utils/huffman.py HuffmanCoding (testing.py:73-76 codes `ids_restore`
 * with it and adds len(bit string) / pixels to the bpp, testing.py:89).  HOST-only (h_ pointers are host memory, nothing
 * touches the device): produces the reference's exact '0'/'1' string, tie-breaking included (CPython heapq on nodes compared
 * by frequency, first-appearance order of the values). */
typedef struct tmae_huffman tmae_huffman;
TMAE_API int  tmae_huffman_create(tmae_huffman** out);
TMAE_API void tmae_huffman_destroy(tmae_huffman* h);
TMAE_API const char* tmae_huffman_last_error(const tmae_huffman* h);
/* HuffmanCoding.compress (utils/huffman.py:141-157): build the code of h_values [n] and encode them; *n_bits = len(encoded_text). */
TMAE_API int  tmae_huffman_compress(tmae_huffman* h, const int64_t* h_values, int64_t n, int64_t* n_bits);
/* The encoded text of the last compress: as_chars = 1 -> one '0' / '1' byte per bit (the reference's Python str, capacity >=
 * n_bits); 0 -> packed, MSB first (capacity >= (n_bits + 7) / 8). */
TMAE_API int  tmae_huffman_bits(const tmae_huffman* h, uint8_t* h_out, int64_t capacity, int as_chars);
/* codes[value] as a NUL-terminated '0'/'1' string. */
TMAE_API int  tmae_huffman_code(const tmae_huffman* h, int64_t value, char* out, int capacity);
/* Distinct values in the key order of the reference's `codes` dict (pre-order walk of the tree); returns their count. */
TMAE_API int  tmae_huffman_num_symbols(const tmae_huffman* h, int64_t* h_values, int64_t capacity);
/* HuffmanCoding.decode (:120-139) with the code of the last compress: *n_values = values decoded. */
TMAE_API int  tmae_huffman_decompress(const tmae_huffman* h, const uint8_t* h_bits, int64_t n_bits, int as_chars,
                             int64_t* h_values, int64_t capacity, int64_t* n_values);

/* Tensor-core GEMM/conv engine self-test hook (tests): C[M,N] = A[M,K] * B[N,K]^T (+bias) with bf16 inputs,
 * run on the tcgen05 kernel (impl 0) or the CUDA-core checker (impl 1). A, B bf16 row-major, C f32. */
TMAE_API int  tmae_gemm_bf16(const void* A, const void* B, const float* bias, float* C, int M, int N, int K,
                    int block_n, int impl, void* stream);
/* C (bf16) = act(A B^T + bias), act = exact-erf GELU when gelu != 0: the bf16 store phases of the engine (QKV / fc1 style layers).
 * variant 0 = one tile per CTA (the one-CTA persistent kernel above two tiles per SM), 1 = CTA pairs, 2 = persistent CTA pairs
 * (double-buffered tensor memory, 74 clusters), 3 = CUDA-core checker. */
TMAE_API int  tmae_gemm_bf16_out(const void* A, const void* B, const float* bias, void* C, int M, int N, int K, int block_n,
                        int gelu, int variant, void* stream);
/* 3x3 pad-1 stride-1 convolution on the engine: x bf16 [N, s, s, Cin] NHWC, w f32 [Cout, Cin, 3, 3] -> f32 NHWC.
 * impl 2 = the CTA-pair (cta_group::2) launch of the tcgen05 kernel. */
TMAE_API int  tmae_conv3x3_bf16(const void* x, const float* w, const float* bias, float* out, int N, int s,
                       int Cin, int Cout, int gelu, int impl, void* stream);

/* Fused softmax attention of the encoder blocks stand-alone (timm Attention.forward, MCM.py:313-322): qkv bf16 [N*T, 3*H*64]
 * with columns [3][H][64] -> out bf16 [N*T, H*64].  impl 0 = mma.sync kernel, 1 = tcgen05 / TMEM kernel (T <= 384), 2 = its
 * multi-stream form (one softmax group per CTA, two CTAs per SM; T <= 96, else the same as 1), 3 = two heads per tile
 * (T = 65 and H even, else the same as 1; measured slower, kept as an experiment). */
TMAE_API int  tmae_attention_bf16(const void* qkv, void* out, int N, int T, int H, int impl, void* stream);
/* The synthesis plan's attention (head dim 32, mma.sync, T up to 1025 and beyond): softmax(q k^T / sqrt(32)) v over qkv bf16
 * [N*T, 3*H*32] with columns [3][H][32] -> out bf16 [N*T, H*32].  Synchronises the stream. */
TMAE_API int  tmae_attention_hd32_bf16(const void* qkv, void* out, int N, int T, int H, void* stream);
/* C = resid + A B^T + bias (fp32 residual in, fp32 out; the proj / fc2 store phase).  pair = 1: the CTA-pair kernel
 * (tcgen05.mma.cta_group::2, 256-row tiles over two SMs; needs block_n % 32 == 0), 0: the one-CTA kernel. */
TMAE_API int  tmae_gemm_bf16_resid(const void* A, const void* B, const float* bias, const float* resid, float* C,
                          int M, int N, int K, int block_n, int pair, int impl, void* stream);
/* The same two self-tests in the precise configurations (TMAE_FLAG_PRECISE_*): fp32 operands, split into `planes` bf16
 * planes inside (2: three tensor-core terms per product, ~1e-5 of an fp32 GEMM / conv; 3: six terms, fp32-equivalent). */
TMAE_API int  tmae_gemm_split(const float* A, const float* B, const float* bias, float* C, int M, int N, int K,
                     int block_n, int planes, int impl, void* stream);
TMAE_API int  tmae_conv3x3_split(const float* x, const float* w, const float* bias, float* out, int N, int s,
                        int Cin, int Cout, int gelu, int planes, int impl, void* stream);

/* Per-kernel-family device timing (bench.py roofline): enable = 1 brackets every launch of tmae_forward with CUDA
 * events on `stream`; enable = 2 brackets every RUN of consecutive launches of one kernel family (keeps the
 * launch-to-launch overlap inside a run, no event gap between its members); 0 = off.  Read after synchronising. */
typedef struct {
    char   name[32];
    int32_t launches;
    float  ms;           /* summed device time */
    double flops;        /* flops of those launches as the reference counts them for the rows actually computed (executed
                            work: patch embed = the K kept patches; 0 for non-GEMM families) */
    double bytes;        /* algorithmic bytes moved (0 if not tracked) */
    double mma_flops;    /* tensor-core flops issued: flops x 3 for precise (split-bf16) layers, else = flops */
} tmae_profile_entry;
TMAE_API int  tmae_profile_enable(tmae_handle* h, int enable);
TMAE_API int  tmae_profile_read(tmae_handle* h, tmae_profile_entry* entries, int max_entries, int* n_entries);
/* Per-launch view of the same events (one entry per plan step, in launch order). */
typedef struct {
    char   name[64];     /* layer tag, e.g. "cc.3.0" */
    float  ms;
    double flops;
    int32_t ctas;        /* CTAs launched (GEMM steps), else 0 */
    int32_t block_n;     /* N tile (GEMM steps), else 0 */
} tmae_profile_step;
TMAE_API int  tmae_profile_read_steps(tmae_handle* h, tmae_profile_step* steps, int max_steps, int* n_steps);
/* Number of kernels tmae_forward launches for batch N (after planning). */
TMAE_API int  tmae_launch_count(tmae_handle* h, int N);

/* Host-only: how the tcgen05 attention kernel is set up for T tokens, H heads, N images in `mode` (1 full form, 2 several
 * streams share the GPU, 3 two-heads-per-tile experiment).  out[12] = {supported (0 -> the mma.sync kernel serves this T), Tp,
 * query tiles, tail rows (computed on CUDA cores), items, S/O/P buffers, pipeline stages, TMEM columns, shared-memory bytes,
 * Q box rows, K/V box rows, form (0 full, 1 lite, 2 duo)}. */
TMAE_API int  tmae_attention_plan(int T, int H, int N, int mode, int* out);

/* Host-only (no device needed): the launch the GEMM engine's policy picks for one GEMM step.
 * shape[17] = {groups, max_M, max_N, conv (0/1), side, n_img, output (0 other, 1 one bf16 same-row output, 2 fp32 same-row
 * output + residual), act (0 none, 1 GELU, 2 0.5 tanh), fused Gaussian (0 none, 1 encoder, 2 decoder), LayerNorm statistics in,
 * LayerNorm statistics out, PixelShuffle output, TMA-store aligned output, share-SM, debug SIMT, forced block_n (0 = policy),
 * forced form (-1 = policy)}; conv shapes need max_M = m_tiles * 128 of tmae_conv_geometry.
 * out[15] = {form (0 one tile per CTA, 1 one-CTA persistent, 2 CTA pairs, 3 persistent CTA pairs, 4 CUDA-core checker), act,
 * store-phase kind, block_n, row tiles, column tiles, grid x, y, z, threads per CTA, dynamic shared memory, pipeline stages,
 * k-blocks per stage, second producer warp, conv A-reuse stage bytes}.  Returns TMAE_EINVAL for an invalid shape or a forced
 * form the shape rules out.  The A/B switches of INTEGRATION.md apply. */
TMAE_API int  tmae_gemm_launch_plan(const int* shape, int* out);

/* Host-only (no device needed): the CTA tiling the conv engine uses for an s x s grid of n_img images.
 * out[6] = {box_y, box_n, y_tiles, m_tiles, rows_used, reuse_ok}.  A tile covers image rows [y0, y0 + box_y) of images
 * [n0, n0 + box_n); rows_used = s * box_y * box_n <= 128 accumulator rows; reuse_ok = the haloed-box A reuse applies
 * (box_n * s is a multiple of the 8-row swizzle atom).  Returns TMAE_EINVAL for s outside 1..128. */
TMAE_API int  tmae_conv_geometry(int s, int n_img, int* out);

#ifdef __cplusplus
}
#endif
#endif /* TMAE_H_ */
