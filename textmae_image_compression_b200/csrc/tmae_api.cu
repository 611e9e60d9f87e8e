// Host runtime behind include/tmae.h: handle, weight ingestion / prepack, per-batch-size launch plans, the forward.
// Every layer of the reference's compression forward path (MCM.py:590-634, 714-787) is one or more entries of a
// static launch plan; tmae_forward only walks the plan (no host sync, no allocation once the plan exists).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/tmae.h"
#include "gemm.cuh"
#include "kernels.h"

using namespace tmae;

namespace {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

std::string g_create_error;

struct RawTensor {
    float* ptr = nullptr;
    std::vector<int64_t> shape;
    size_t numel = 0;
};

struct Layer {                      // one prepacked linear / conv
    __nv_bfloat16* w = nullptr;     // [Cout, Kp]
    float* bias = nullptr;          // [Cout] (permuted for PixelShuffle layers)
    int Cout = 0, Cin = 0, taps = 1, nseg = 1, segc[3] = {0, 0, 0}, Kp = 0, shuffle = 0;
    float* wsum = nullptr;          // LayerNorm folded into this linear (W' = W diag(gamma), bias' = bias + W beta): row sums of bf16(W')
    int planes = 1;                 // 2 / 3 = precise layer: every tap holds the hi planes of its segments, then the lo (mid, lo) planes
    int kb_tap = 0;                 // k-blocks of one plane of one tap
};

// bf16 activation buffer of the workspace; `lo` = plane layout when the layer that reads it is precise (split-bf16):
// 0 one plane, > 0 two planes `lo` elements apart, < 0 three planes `-lo` apart (store_bf16x4_planes in common.cuh)
struct Bf {
    __nv_bfloat16* p = nullptr;
    long long lo = 0;
};

enum StepKind { ST_MASK, ST_GATHER, ST_GEMM, ST_FORCE, ST_LN, ST_ATTN, ST_EB, ST_GC, ST_RATE, ST_ZERO_RATE,
                ST_ZDEQ, ST_IDX, ST_YDEQ, ST_DEC_OUT,        // decode plans only
                ST_ZDEC, ST_YDEC,                            // decode-from-streams plans only: the range decoder
                ST_SYN_IN, ST_UNSHUF, ST_ATTN32, ST_UNPATCH };  // synthesis plans only
enum Family { FAM_GEMM = 0, FAM_ATTN, FAM_LN, FAM_MASK, FAM_GATHER, FAM_ENTROPY, FAM_MISC, FAM_CODER, FAM_COUNT };
const char* kFamilyNames[FAM_COUNT] = {"gemm_tc", "attention", "layernorm", "mask_select", "gather_patches",
                                       "entropy_elementwise", "misc", "entropy_coder"};

struct Step {
    StepKind kind;
    int family = FAM_MISC;
    // GEMM
    int param_index = 0, groups = 1, max_M = 0, max_N = 0, block_n = 0, act = 0, epi = 0;
    int next_index = -1, next_groups = 0;      // parameter blocks of the next GEMM step (weight prefetch target)
    int conv_reuse_stage_bytes = 0;            // > 0: 3x3 conv launch with haloed-box A reuse, stage size in bytes
    bool pair = false;                         // CTA-pair (cta_group::2) launch
    bool pair_persist = false;                 // ... as the persistent pair kernel (one batch in flight, several tiles per cluster)
    double flops = 0, bytes = 0;
    int mma_terms = 1;                         // 3 for precise (split-bf16) GEMM steps
    // LN
    const float* ln_gamma = nullptr;
    const float* ln_beta = nullptr;
    int ln_final = 0;
    // GC
    int slice = 0, gc_slices = 1;
    // ST_ZDEC / ST_YDEC: lanes per stream (0 = compressai's format)
    int lanes = 0;
    std::string tag;
};

// Plan kinds, and what each kind's steps and captured graphs read.  drop_plans(h, DEP_x) discards every plan that reads x
// when x is freed or rewritten; the next call of that kind builds its plan again.
enum PlanKind {
    PLAN_FORWARD,                    // tmae_forward and the calls that run part of it
    PLAN_FORCED,                     // tmae_forward_from_latent_forced
    PLAN_DECODE,                     // tmae_decode_begin / _step
    PLAN_STREAMS,                    // tmae_decompress_streams(_lanes): the decode with the range decoder in front
    PLAN_SYNTH,                      // tmae_synthesize
};
enum PlanDep : unsigned {
    DEP_WS = 1,                      // network workspace (ensure_workspace)
    DEP_CODER = 2,                   // coder workspace (ensure_coder_workspace)
    DEP_SYNTH = 4,                   // synthesis workspace (ensure_synth_workspace, tmae_enable_synthesis)
    DEP_SCALE = 8,                   // scale table (tmae_set_scale_table)
    DEP_CDF = 16,                    // CDF tables (tmae_set_cdf_tables)
    DEP_ALL = ~0u,                   // weights (tmae_finalize_weights) and tmae_destroy: every plan
};
const unsigned kPlanDeps[] = {
    DEP_WS | DEP_SCALE,                          // PLAN_FORWARD
    DEP_WS | DEP_SCALE,                          // PLAN_FORCED
    DEP_WS | DEP_SCALE,                          // PLAN_DECODE
    DEP_WS | DEP_SCALE | DEP_CODER | DEP_CDF,    // PLAN_STREAMS
    DEP_SYNTH,                                   // PLAN_SYNTH
};
// (kind, batch size, y lanes, z lanes); the lanes are nonzero for the laned PLAN_STREAMS only
typedef std::tuple<int, int, int, int> PlanKey;

struct Plan {
    int N = 0;
    unsigned deps = 0;               // DEP_* bits of its kind
    std::vector<Step> steps;
    std::vector<GemmParams> host_params;
    GemmParams* d_params = nullptr;
    bool from_latent_ok = true;
    bool attn_tc = false;           // tcgen05 attention: tensor maps of the Q and K / V tiles over this plan's qkv matrix
    CUtensorMap attn_q, attn_k;
    int first_rate_step = 0;        // index of the first step of the rate half (h_a)
    int encoder_end_step = 0;       // one past the final LayerNorm
    // stage k = steps [stage_begin[k], stage_begin[k + 1]), one CUDA graph per stage (run_stage).  Builders add the cuts
    // (the step-wise decode only); finish_plan closes the last stage.
    std::vector<int> stage_begin{0};
    std::vector<cudaGraphExec_t> stage_graph;
    std::vector<int> stage_calls;

    Plan() = default;
    Plan(const Plan&) = delete;
    Plan& operator=(const Plan&) = delete;
    ~Plan() {
        if (d_params) cudaFree(d_params);
        for (cudaGraphExec_t g : stage_graph) if (g) cudaGraphExecDestroy(g);
    }
};

struct Workspace {
    int cap_N = 0;
    size_t bytes = 0;
    std::vector<void*> allocs;
    // encoder
    int64_t* ids_keep = nullptr;
    Bf patches, xn, qkv, attn, h1, enc;
    Bf x_bf;                         // bf16 copy of the residual stream (A operand of the LayerNorm-folded QKV / fc1)
    float* ln_stats = nullptr;       // [2 * depth][N * T][C / 32][2]: (sum x, sum x^2) partials per LayerNorm, token and 32-column chunk
    float* x = nullptr;
    // g_a
    Bf ga1, ga2, ga3, y_bf;
    float *y = nullptr, *z = nullptr, *mu = nullptr, *sigma = nullptr, *yhat = nullptr;
    float* yhat_force = nullptr;     // slice-wise teacher forcing: the caller's y_hat (support of every later slice)
    // h_a / h_s
    Bf ha1, ha2, ha3, ha4, zhat_bf;
    Bf hs1[2], hs2[2], hs3[2], hs4[2], lat[2];     // 0 = means, 1 = scales
    Bf yhat_bf;
    Bf t[18][4];                                   // [slice-group member j (0..5) * 3 + net (mean, scale, lrp)][layer]
    double* rate_acc = nullptr;
    float* bpp = nullptr;
    double* rate_sums = nullptr;
    // host-buffer entry staging
    float *st_imgs = nullptr, *st_scores = nullptr;
    float *st_ylik = nullptr, *st_zlik = nullptr;          // device staging of the host-returned results (tmae_forward_host)
    int16_t *st_ysym = nullptr, *st_zsym = nullptr;
    int64_t* st_ids_restore = nullptr;
    IoBlock* io = nullptr;           // per-call pointers for graph replays
};

// Buffers of the entropy coder, grown on demand apart from the network's workspace (a forward-only handle never needs them).
struct CoderWorkspace {
    std::vector<void*> allocs;
    int cap_N = 0;                   // decode from streams: batch capacity of the four buffers below
    int32_t* zsym = nullptr;         // [N, Cz, s/4, s/4] decoded z symbols (ST_ZDEC -> ST_ZDEQ)
    int32_t* ysym = nullptr;         // [N, Cy * K] decoded y symbols (ST_YDEC -> ST_YDEQ)
    int32_t* idx = nullptr;          // [N, Cy * K] scale-table indexes, when the caller does not ask for them
    RansDecState* state = nullptr;   // [N * 32] y decoder state between the slice groups (per image, or per image and lane)
    size_t enc_bytes = 0;            // tmae_rans_encode scratch: records, per-stream word regions, word counts
    void* enc = nullptr;
};

// Buffers of the synthesis plans (tmae_synthesize), allocated only on handles with synthesis enabled.  All bf16 buffers hold
// one plane: synthesis runs bf16 operands in every accuracy mode.
struct SynthWorkspace {
    std::vector<void*> allocs;
    int cap_N = 0;
    Bf y_bf;                         // [N*K, Cy] the caller's y_hat in bf16 (A operand of g_s.0)
    Bf gs[3], tok;                   // g_s.0 / .2 / .4 outputs, g_s.6 output [N*K, E]
    float* emb = nullptr;            // decoder_embed output [N*K, Dd]
    float* x = nullptr;              // residual stream of the MAE decoder [N*T, Dd], T = L + 1
    Bf x_bf, qkv, attn, h1, pred;    // pred: decoder_pred output [N*T, p*p*3]
    float* ln_stats = nullptr;       // [2 * depth + 1][N * T][Dd / 32][2]: norm1 / norm2 of every block, then decoder_norm
    IoBlock* io = nullptr;           // per-call pointers (y_hat, ids_restore, x_hat)
};

// One profiled launch, or one run of consecutive same-family launches (tmae_profile_enable(h, 2)).
struct ProfRecord {
    cudaEvent_t begin = nullptr, end = nullptr;
    int family = 0;
    double flops = 0, bytes = 0, mma_flops = 0;
    std::string tag;                 // the first step's tag
    int ctas = 0, block_n = 0;       // the first step's GEMM grid and tile width (0: not a GEMM)
    int launches = 0;
};

}  // namespace

struct tmae_handle {
    tmae_config cfg;
    int L, K, T, s, C, H, hd, mlp, Cy, Cz, nsl, sc, grid_w, patch_dim, s2, s4;
    int ga_ch[5];
    std::string err;
    std::map<std::string, RawTensor> raw;
    std::map<std::string, Layer> layers;
    std::map<std::string, float*> vecs;       // fp32 vectors kept as-is (LN params, cls, pos-embed)
    float* eb_tab = nullptr;
    float* scale_table = nullptr;    // GaussianConditional scale table (tmae_set_scale_table) for y_indexes
    int n_scale_table = 0;
    bool gc_fuse = false;            // bf16 rate half: cc_transform_mean/scale[i].8 as one GEMM with the Gaussian conditional in its epilogue
    bool finalized = false;
    Workspace ws;
    std::map<PlanKey, std::unique_ptr<Plan>> plans;   // every launch plan of the handle (get_plan)
    // synthesis (tmae_enable_synthesis): g_s, the MAE decoder and unpatchify on the engine
    int syn_depth = 0, syn_heads = 0;    // 0: synthesis disabled (the decoder-side weights are ignored)
    int Dd = 0, syn_mlp = 0, syn_out = 0; // decoder width, its MLP width, decoder_pred outputs (p * p * in_chans)
    SynthWorkspace sws;
    CdfTables cdf[2];                // quantised CDF tables: [TMAE_MODEL_GAUSSIAN], [TMAE_MODEL_BOTTLENECK]
    CoderWorkspace cws;
    int dec_N = 0, dec_next = -1;    // decode in progress: batch size and the next group expected (-1 = none)
    PFN_encodeTiled encode = nullptr;
    std::vector<void*> weight_allocs;
    bool use_graph = true;           // TMAE_NO_GRAPH=1 disables CUDA-graph replay
    bool precise_rate = false;       // TMAE_FLAG_PRECISE_RATE / _ALL: split-bf16 layers after the encoder
    bool precise_enc = false;        // TMAE_FLAG_PRECISE_ALL: the encoder as well
    bool ln_fold = false;            // bf16 encoder: LayerNorm of the blocks folded into proj / fc2 (statistics) and QKV / fc1 (apply)
    int planes = 2;                  // bf16 planes per operand of a precise layer: 2 (3 terms) or 3 (TMAE_FLAG_PRECISE_X6, 6 terms)
    cudaStream_t cap_stream = nullptr;
    // profiling
    bool profiling = false;
    bool prof_by_run = false;        // one event pair per run of consecutive same-family launches instead of per launch
    std::vector<ProfRecord> prof;    // records of the profiled call; the events are kept for the next one
    size_t prof_used = 0;
    int dev = 0;
};

namespace {

int fail(tmae_handle* h, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CUDA_TRY(h, expr)                                                                          \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail((h), TMAE_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

template <typename Tp>
int dev_alloc(tmae_handle* h, std::vector<void*>& pool, Tp** out, size_t count, size_t* total = nullptr) {
    void* p = nullptr;
    size_t bytes = count * sizeof(Tp);
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return fail(h, TMAE_ENOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    e = cudaMemset(p, 0, bytes);
    if (e != cudaSuccess) return fail(h, TMAE_ECUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    pool.push_back(p);
    *out = reinterpret_cast<Tp*>(p);
    if (total) *total += bytes;
    return TMAE_OK;
}

int pad64(int c) { return (c + 63) / 64 * 64; }
int round16(int c) { return (c + 15) / 16 * 16; }

// ---- geometry ------------------------------------------------------------------------------------------
int derive_geometry(tmae_handle* h) {
    const tmae_config& c = h->cfg;
    if (c.img_size <= 0 || c.patch_size <= 0 || c.img_size % c.patch_size != 0)
        return fail(nullptr, TMAE_EINVAL, "image size %d must be a positive multiple of patch size %d", c.img_size, c.patch_size);
    h->grid_w = c.img_size / c.patch_size;
    h->L = h->grid_w * h->grid_w;
    h->K = c.num_keep_patches;
    if (h->K > h->L)
        return fail(nullptr, TMAE_EINVAL, "Number of patches should not be greater than the length of scores");   // MCM.py:374-376
    h->s = (int)lround(sqrt((double)h->K));
    if (h->s * h->s != h->K)
        return fail(nullptr, TMAE_EINVAL, "num_keep_patches=%d is not a perfect square (reference view() at MCM.py:729 fails)", h->K);
    if (h->s % 4 != 0)
        return fail(nullptr, TMAE_EINVAL, "sqrt(num_keep_patches)=%d must be a multiple of 4 (reference torch.cat at MCM.py:761 fails)", h->s);
    h->T = h->K + 1;
    h->C = c.encoder_embed_dim;
    h->H = c.encoder_num_heads;
    if (h->H <= 0 || h->C % h->H != 0 || h->C / h->H != 64)
        return fail(nullptr, TMAE_EINVAL, "head_dim must be 64 (embed %d / heads %d)", h->C, h->H);
    h->hd = 64;
    h->mlp = (int)(h->C * c.mlp_ratio);
    h->Cy = c.latent_depth;
    h->Cz = c.hyperprior_depth;
    h->nsl = c.num_slices;
    if (h->nsl != 12 || h->Cy % h->nsl != 0 || (h->Cy / h->nsl) % 8 != 0)
        return fail(nullptr, TMAE_EINVAL, "unsupported latent_depth/num_slices %d/%d", h->Cy, h->nsl);
    h->sc = h->Cy / h->nsl;
    h->patch_dim = c.in_chans * c.patch_size * c.patch_size;
    if (c.patch_size % 4 != 0 || h->C % 128 != 0)
        return fail(nullptr, TMAE_EINVAL, "patch_size %% 4 and embed_dim %% 128 required");
    h->s2 = h->s / 2;
    h->s4 = h->s / 4;
    const int e = h->C, d = c.decoder_embed_dim;
    h->ga_ch[0] = e;
    h->ga_ch[1] = (int)(d + (e - d) * 3 / 4.0);
    h->ga_ch[2] = (int)(d + (e - d) * 2 / 4.0);
    h->ga_ch[3] = d;
    h->ga_ch[4] = h->Cy;
    for (int i = 0; i < 5; ++i)
        if (h->ga_ch[i] % 8 != 0) return fail(nullptr, TMAE_EINVAL, "g_a channel %d not a multiple of 8", h->ga_ch[i]);
    return TMAE_OK;
}

void ha_layers(const tmae_handle* h, int cin[5], int cout[5], int stride[5]) {
    const int m = h->Cy, z = h->Cz;
    const int c1 = (int)(z + (m - z) * 3 / 4.0), c2 = (int)(z + (m - z) * 2 / 4.0), c3 = (int)(z + (m - z) / 4.0);
    const int ci[5] = {m, m, c1, c2, c3}, co[5] = {m, c1, c2, c3, z}, st[5] = {1, 1, 2, 1, 2};
    for (int i = 0; i < 5; ++i) { cin[i] = ci[i]; cout[i] = co[i]; stride[i] = st[i]; }
}
void hs_layers(const tmae_handle* h, int cin[5], int cout[5], int up[5]) {
    const int m = h->Cy, z = h->Cz;
    const int c1 = (int)(z + (m - z) / 4.0), c2 = (int)(z + (m - z) * 2 / 4.0), c3 = (int)(z + (m - z) * 3 / 4.0);
    const int ci[5] = {z, c1, c2, c3, m}, co[5] = {c1, c2, c3, m, m}, u[5] = {1, 2, 1, 2, 1};
    for (int i = 0; i < 5; ++i) { cin[i] = ci[i]; cout[i] = co[i]; up[i] = u[i]; }
}
void cc_channels(const tmae_handle* h, int ch[6], int i, bool lrp) {
    const int sc = h->sc, ns = h->nsl;
    const int sup = lrp ? (i + 1 < ns / 2 + 1 ? i + 1 : ns / 2 + 1) : (i < ns / 2 ? i : ns / 2);
    ch[0] = h->Cy + sc * sup;
    ch[1] = (int)(sc * (ns / 2 + 1));
    ch[2] = (int)(sc * (ns / 2 * 3 / 4.0 + 1));
    ch[3] = (int)(sc * (ns / 2 * 2 / 4.0 + 1));
    ch[4] = (int)(sc * (ns / 2 * 1 / 4.0 + 1));
    ch[5] = sc;
}

// ---- weights -------------------------------------------------------------------------------------------
bool name_is_needed(const tmae_handle* h, const std::string& n) {
    static const char* prefixes[] = {"cls_token", "encoder_pos_embed", "encoder_embed.", "encoder_blocks.",
                                     "encoder_norm.", "g_a.", "h_a.", "h_s_mean.", "h_s_scale.", "cc_transform_mean.",
                                     "cc_transform_scale.", "lrp_transform.", "entropy_bottleneck._matrix",
                                     "entropy_bottleneck._bias", "entropy_bottleneck._factor",
                                     "entropy_bottleneck.quantiles"};
    static const char* decoder_prefixes[] = {"g_s.", "decoder_embed.", "mask_token", "decoder_pos_embed", "decoder_blocks.",
                                             "decoder_norm.", "decoder_pred."};
    for (const char* p : prefixes)
        if (n.compare(0, strlen(p), p) == 0) return true;
    if (h->syn_depth > 0)                    // synthesis enabled: the decoder side is needed as well
        for (const char* p : decoder_prefixes)
            if (n.compare(0, strlen(p), p) == 0) return true;
    return false;
}

const RawTensor* find_raw(tmae_handle* h, const std::string& name) {
    auto it = h->raw.find(name);
    return it == h->raw.end() ? nullptr : &it->second;
}

int need_raw(tmae_handle* h, const std::string& name, size_t numel, const RawTensor** out) {
    const RawTensor* r = find_raw(h, name);
    if (!r) return fail(h, TMAE_ESTATE, "missing weight '%s'", name.c_str());
    if (r->numel != numel)
        return fail(h, TMAE_EINVAL, "weight '%s' has %zu elements, expected %zu", name.c_str(), r->numel, numel);
    *out = r;
    return TMAE_OK;
}

// Prepack one conv / linear: weight [Cout, Cin, taps] fp32 -> bf16 [Cout, Kp]; bias fp32 (permuted if shuffle).
int pack_layer(tmae_handle* h, const std::string& key, const std::string& wname, int Cout, int Cin, int taps, int nseg,
               const int* segc, int shuffle, bool precise, const std::string& fold_ln = std::string()) {
    const RawTensor *w = nullptr, *b = nullptr;
    int rc = need_raw(h, wname + ".weight", (size_t)Cout * Cin * taps, &w);
    if (rc) return rc;
    rc = need_raw(h, wname + ".bias", (size_t)Cout, &b);
    if (rc) return rc;
    {   // layout check, not only the element count: [Cout, Cin] / [Cout, Cin, k, k] (a transposed tensor must not pass)
        const std::vector<int64_t>& sh = w->shape;
        const int k = taps == 9 ? 3 : 0;
        bool ok = sh.size() >= 2 && sh[0] == Cout;
        if (ok && taps == 9) ok = sh.size() == 4 && sh[1] == Cin && sh[2] == k && sh[3] == k;
        if (ok && taps == 1) { int64_t rest = 1; for (size_t i = 1; i < sh.size(); ++i) rest *= sh[i]; ok = rest == Cin && (sh.size() == 2 || sh.size() == 4); }
        if (!ok) return fail(h, TMAE_EINVAL, "weight '%s.weight' has the wrong shape (expected [%d, %d%s])", wname.c_str(), Cout, Cin,
                             taps == 9 ? ", 3, 3" : "");
    }
    Layer L;
    L.Cout = Cout; L.Cin = Cin; L.taps = taps; L.nseg = nseg; L.shuffle = shuffle;
    int kp_tap = 0, csum = 0;
    for (int i = 0; i < nseg; ++i) { L.segc[i] = segc[i]; kp_tap += pad64(segc[i]); csum += segc[i]; }
    if (csum != Cin) return fail(h, TMAE_EINVAL, "layer %s: segments sum %d != Cin %d", key.c_str(), csum, Cin);
    L.planes = precise ? h->planes : 1;
    L.kb_tap = kp_tap / 64;
    L.Kp = kp_tap * taps * L.planes;
    rc = dev_alloc(h, h->weight_allocs, &L.w, (size_t)Cout * L.Kp);
    if (rc) return rc;
    rc = dev_alloc(h, h->weight_allocs, &L.bias, (size_t)Cout);
    if (rc) return rc;
    if (!fold_ln.empty()) {            // LayerNorm `fold_ln` (.weight / .bias) folded into this linear layer
        const RawTensor *g = nullptr, *be = nullptr;
        if (taps != 1 || nseg != 1 || shuffle || precise) return fail(h, TMAE_EINVAL, "layer %s: LayerNorm fold needs a plain bf16 linear", key.c_str());
        if ((rc = need_raw(h, fold_ln + ".weight", (size_t)Cin, &g)) || (rc = need_raw(h, fold_ln + ".bias", (size_t)Cin, &be))) return rc;
        if ((rc = dev_alloc(h, h->weight_allocs, &L.wsum, (size_t)Cout))) return rc;
        CUDA_TRY(h, launch_prepack_weight(w->ptr, L.w, Cout, Cin, taps, nseg, L.segc, shuffle, L.planes, 0, g->ptr));
        CUDA_TRY(h, launch_fold_ln(w->ptr, be->ptr, b->ptr, L.w, L.Kp, Cout, Cin, L.bias, L.wsum, 0));
        h->layers[key] = L;
        return TMAE_OK;
    }
    CUDA_TRY(h, launch_prepack_weight(w->ptr, L.w, Cout, Cin, taps, nseg, L.segc, shuffle, L.planes, 0));
    if (shuffle) CUDA_TRY(h, launch_permute_bias_shuffle(b->ptr, L.bias, Cout, 0));
    else CUDA_TRY(h, cudaMemcpyAsync(L.bias, b->ptr, (size_t)Cout * sizeof(float), cudaMemcpyDeviceToDevice, 0));
    h->layers[key] = L;
    return TMAE_OK;
}

int keep_vec(tmae_handle* h, const std::string& name, size_t numel) {
    const RawTensor* r = nullptr;
    int rc = need_raw(h, name, numel, &r);
    if (rc) return rc;
    float* p = nullptr;
    rc = dev_alloc(h, h->weight_allocs, &p, numel);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(p, r->ptr, numel * sizeof(float), cudaMemcpyDeviceToDevice, 0));
    h->vecs[name] = p;
    return TMAE_OK;
}

// Decoder side of the weights (tmae_enable_synthesis), bf16 in every accuracy mode.  g_s.<l> are ConvTranspose2d 1x1 weights
// [cin, cout, 1, 1]: transposed to [cout, cin] here, then packed like every linear.  The block LayerNorms and decoder_norm are
// folded into the layers that read them (QKV, fc1, decoder_pred).
int pack_synthesis(tmae_handle* h) {
    const int Dd = h->Dd, T = h->L + 1;
    int rc;
    const int ch[5] = {h->Cy, h->ga_ch[3], h->ga_ch[2], h->ga_ch[1], h->C};
    for (int l = 0; l < 4; ++l) {
        const std::string nm = "g_s." + std::to_string(2 * l);
        const RawTensor *w = nullptr, *b = nullptr;
        if ((rc = need_raw(h, nm + ".weight", (size_t)ch[l] * ch[l + 1], &w)) || (rc = need_raw(h, nm + ".bias", (size_t)ch[l + 1], &b))) return rc;
        if (w->shape.size() != 4 || w->shape[0] != ch[l] || w->shape[1] != ch[l + 1] || w->shape[2] != 1 || w->shape[3] != 1)
            return fail(h, TMAE_EINVAL, "weight '%s.weight' has the wrong shape (expected ConvTranspose2d [%d, %d, 1, 1])", nm.c_str(), ch[l], ch[l + 1]);
        std::vector<float> src(w->numel), dst(w->numel), bias(b->numel);
        CUDA_TRY(h, cudaMemcpy(src.data(), w->ptr, w->numel * sizeof(float), cudaMemcpyDeviceToHost));
        CUDA_TRY(h, cudaMemcpy(bias.data(), b->ptr, b->numel * sizeof(float), cudaMemcpyDeviceToHost));
        for (int i = 0; i < ch[l]; ++i)
            for (int o = 0; o < ch[l + 1]; ++o) dst[(size_t)o * ch[l] + i] = src[(size_t)i * ch[l + 1] + o];
        RawTensor wt, bt;
        wt.numel = w->numel; wt.shape = {ch[l + 1], ch[l]};
        bt.numel = b->numel; bt.shape = {ch[l + 1]};
        CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&wt.ptr), wt.numel * sizeof(float)));
        h->raw[nm + ".T.weight"] = wt;          // freed with the other raw tensors at the end of finalize
        CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&bt.ptr), bt.numel * sizeof(float)));
        h->raw[nm + ".T.bias"] = bt;
        CUDA_TRY(h, cudaMemcpy(wt.ptr, dst.data(), wt.numel * sizeof(float), cudaMemcpyHostToDevice));
        CUDA_TRY(h, cudaMemcpy(bt.ptr, bias.data(), bt.numel * sizeof(float), cudaMemcpyHostToDevice));
        int sg[1] = {ch[l]};
        if ((rc = pack_layer(h, nm, nm + ".T", ch[l + 1], ch[l], 1, 1, sg, 0, false))) return rc;
    }
    { int sg[1] = {h->C}; if ((rc = pack_layer(h, "decoder_embed", "decoder_embed", Dd, h->C, 1, 1, sg, 0, false))) return rc; }
    const RawTensor* r = nullptr;
    if ((rc = need_raw(h, "mask_token", (size_t)Dd, &r))) return rc;
    if (r->shape.size() != 3 || r->shape[0] != 1 || r->shape[1] != 1)
        return fail(h, TMAE_EINVAL, "weight 'mask_token' has the wrong shape (expected [1, 1, %d])", Dd);
    if ((rc = need_raw(h, "decoder_pos_embed", (size_t)T * Dd, &r))) return rc;
    if (r->shape.size() != 3 || r->shape[0] != 1 || r->shape[1] != T || r->shape[2] != Dd)
        return fail(h, TMAE_EINVAL, "weight 'decoder_pos_embed' has the wrong shape (expected [1, %d, %d])", T, Dd);
    if ((rc = keep_vec(h, "mask_token", Dd)) || (rc = keep_vec(h, "decoder_pos_embed", (size_t)T * Dd))) return rc;
    for (int i = 0; i < h->syn_depth; ++i) {
        const std::string pre = "decoder_blocks." + std::to_string(i);
        int sgD[1] = {Dd}, sgM[1] = {h->syn_mlp};
        if ((rc = pack_layer(h, pre + ".attn.qkv", pre + ".attn.qkv", 3 * Dd, Dd, 1, 1, sgD, 0, false, pre + ".norm1")) ||
            (rc = pack_layer(h, pre + ".attn.proj", pre + ".attn.proj", Dd, Dd, 1, 1, sgD, 0, false)) ||
            (rc = pack_layer(h, pre + ".mlp.fc1", pre + ".mlp.fc1", h->syn_mlp, Dd, 1, 1, sgD, 0, false, pre + ".norm2")) ||
            (rc = pack_layer(h, pre + ".mlp.fc2", pre + ".mlp.fc2", Dd, h->syn_mlp, 1, 1, sgM, 0, false)))
            return rc;
    }
    int sg[1] = {Dd};
    return pack_layer(h, "decoder_pred", "decoder_pred", h->syn_out, Dd, 1, 1, sg, 0, false, "decoder_norm");
}

// ---- tensor maps ---------------------------------------------------------------------------------------
int make_map(tmae_handle* h, CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems,
             uint32_t box_rows) {
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {ld_elems * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBlockK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    if (rows == 0 || cols == 0) return fail(h, TMAE_EINVAL, "empty tensor map");
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (gstr[0] & 15) != 0)
        return fail(h, TMAE_EINVAL, "tensor map base/stride not 16-byte aligned");
    CUresult r = h->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(h, TMAE_ECUDA, "cuTensorMapEncodeTiled failed (%d): cols %llu rows %llu ld %llu box_rows %u", (int)r,
                    (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)ld_elems, box_rows);
    return TMAE_OK;
}

// Output of the TMA-store epilogue: [rows, cols] bf16 row-major, box = 32 columns x 128 rows, SWIZZLE_64B (64-byte rows).
int make_store_map(tmae_handle* h, CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems) {
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {ld_elems * 2};
    cuuint32_t box[2] = {32, (cuuint32_t)kBlockM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = h->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(h, TMAE_ECUDA, "cuTensorMapEncodeTiled(store) failed (%d): cols %llu rows %llu ld %llu", (int)r,
                    (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)ld_elems);
    return TMAE_OK;
}

// Conv A operand: the compact channels-last tensor [n_img, s, s, C] seen as a 4-D tensor (C, x, n, y); one box is
// [64 ch, s, box_n, rows_y] = s * box_n * rows_y rows of 128 B in smem (row = (yl * box_n + nl) * s + x), SWIZZLE_128B.
// rows_y = box_y, or box_y + 2 for the haloed box of conv_reuse.
int make_map4d(tmae_handle* h, CUtensorMap* map, const void* base, uint64_t cols, int s, int n_img, uint64_t ld_elems,
               int box_n, int rows_y, uint32_t box_cols = kBlockK, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    cuuint64_t gdim[4] = {cols, (cuuint64_t)s, (cuuint64_t)n_img, (cuuint64_t)s};
    cuuint64_t gstr[3] = {ld_elems * 2, (cuuint64_t)s * s * ld_elems * 2, (cuuint64_t)s * ld_elems * 2};
    cuuint32_t box[4] = {box_cols, (cuuint32_t)s, (cuuint32_t)box_n, (cuuint32_t)rows_y};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if (cols == 0 || s <= 0 || n_img <= 0) return fail(h, TMAE_EINVAL, "empty tensor map");
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (gstr[0] & 15) != 0)
        return fail(h, TMAE_EINVAL, "tensor map base/stride not 16-byte aligned");
    CUresult r = h->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(h, TMAE_ECUDA, "cuTensorMapEncodeTiled(4d) failed (%d): cols %llu s %d n %d ld %llu box %d x %d", (int)r,
                    (unsigned long long)cols, s, n_img, (unsigned long long)ld_elems, box_n, rows_y);
    return TMAE_OK;
}

// Tiling of a conv layer over an s x s grid: a CTA tile is box_y image rows of box_n images (s * box_y * box_n <= 128
// accumulator rows).  Pick the pair with the fewest tiles.  A pair whose dy shift (box_n * s rows) is a whole number of
// 8-row swizzle atoms can use the haloed-box A reuse (GemmParams::conv_reuse); such a pair wins unless it costs more
// than 15 % extra tiles.
struct ConvGeom { int box_y = 0, box_n = 0, y_tiles = 0, m_tiles = 0, rows_used = 0; bool reuse_ok = false; };
bool conv_geom(int s, int n_img, ConvGeom* g) {
    if (s <= 0 || s > kBlockM || n_img <= 0) return false;
    long long best[2] = {-1, -1};          // [0] any pair, [1] reuse-compatible pair
    ConvGeom cand[2];
    for (int by = (s < kBlockM / s ? s : kBlockM / s); by >= 1; --by) {
        for (int pass = 0; pass < 2; ++pass) {
            int bn = kBlockM / (s * by);
            if (bn > 256) bn = 256;
            if (pass == 0) { if (bn > n_img) bn = n_img; }
            else {
                int q = 8; for (int d = 8; d >= 1; d >>= 1) if (s % d == 0) { q = 8 / d; break; }   // q = 8 / gcd(s, 8)
                bn = bn / q * q;                                   // box_n * s must be a multiple of 8 rows
                while (bn - q >= n_img && bn - q > 0) bn -= q;     // no more images per tile than needed
                if (by < 2) bn = 0;                                // one row + two halo rows: nothing to reuse
            }
            if (bn <= 0) continue;
            const int yt = (s + by - 1) / by;
            const long long tiles = (long long)((n_img + bn - 1) / bn) * yt;
            if (best[pass] < 0 || tiles < best[pass]) {
                best[pass] = tiles;
                cand[pass].box_y = by; cand[pass].box_n = bn; cand[pass].y_tiles = yt; cand[pass].m_tiles = (int)tiles;
                cand[pass].rows_used = s * by * bn; cand[pass].reuse_ok = pass == 1;
            }
        }
    }
    if (best[0] < 0) return false;
    static const bool no_reuse = getenv("TMAE_NO_CONV_REUSE") != nullptr;
    *g = (!no_reuse && best[1] > 0 && best[1] * 100 <= best[0] * 115) ? cand[1] : cand[0];
    return true;
}

// Choose the N tile: fewest column tiles that still give the machine >= ~120 CTAs (148 SMs), multiple of 16.
int pick_block_n(int m_tiles, int N, int groups) {
    int best = round16(N) > 256 ? 256 : round16(N);
    for (int nt = 1; nt <= 16; ++nt) {
        int bn = round16((N + nt - 1) / nt);
        if (bn > 256) continue;
        best = bn;
        if ((long long)m_tiles * nt * groups >= 120 || bn <= 64) break;
    }
    return best;
}

struct SegSrc {
    const __nv_bfloat16* ptr;   // first column of the segment
    int cols;                   // channels in the segment
    int ld;                     // row pitch (elements)
    long long lo;               // element offset of the lo plane (precise layers), else 0
};

struct GemmDesc {
    const Layer* layer = nullptr;
    SegSrc seg[3];
    int nseg = 1;
    long long a_rows = 0;       // rows of the A matrices
    int M = 0;                  // rows to compute
    int in_mode = IN_LINEAR;
    int side = 0;               // grid side for IN_COMPACT / IN_CONV
    int n_img = 0;              // IN_CONV: images
    bool conv_reuse = false;    // IN_CONV: haloed-box A reuse (decided per launch in add_gemm_group)
    bool conv3 = false;
    int act = ACT_NONE;
    const float* resid = nullptr; int resid_ld = 0; int resid_map = MAP_SAME;
    const int64_t* gather_ids = nullptr;
    const float* ln_stats_in = nullptr;     // folded LayerNorm, consumer side (the layer's pack carries gamma / beta / wsum)
    float* ln_stats_out = nullptr;          // producer side: statistics + bf16 copy of the output rows
    __nv_bfloat16* xbf_out = nullptr;
    OutSpec out0 = {nullptr, 0, OUT_NONE, MAP_SAME, 0};
    OutSpec out1 = {nullptr, 0, OUT_NONE, MAP_SAME, 0};
    double flops = 0;
    int gc_slice = -1;          // >= 0: fused mean + scale last layer of this slice, Gaussian conditional in the epilogue
    bool gc_decode = false;     // ... decoder form: mu, sigma and scale-table indexes only (EPI_GAUSS_IDX)
};

int fill_params(tmae_handle* h, const GemmDesc& d, int groups_for_tiling, GemmParams* p, int force_block_n) {
    memset(p, 0, sizeof(*p));
    const Layer& L = *d.layer;
    if (d.nseg != L.nseg) return fail(h, TMAE_EINVAL, "segment count mismatch");
    const bool conv = d.in_mode == IN_CONV;
    if (conv != (L.taps == 9)) return fail(h, TMAE_EINVAL, "3x3 layers need IN_CONV inputs (and only they)");
    ConvGeom cg;
    if (conv) {
        if (!conv_geom(d.side, d.n_img, &cg)) return fail(h, TMAE_EINVAL, "conv grid side %d unsupported (1..128)", d.side);
        if (d.M != cg.m_tiles * kBlockM || d.a_rows != (long long)d.n_img * d.side * d.side)
            return fail(h, TMAE_EINVAL, "conv descriptor rows inconsistent with its geometry");
    }
    // K segments: one per concatenated source; a precise layer issues several split-bf16 terms per source, each one more
    // segment (activation plane pa x weight plane pw): 2 planes -> hi*hi, lo*hi, hi*lo; 3 planes -> + mid*mid, lo*hi, hi*lo
    static const int kTerms2[3][2] = {{0, 0}, {1, 0}, {0, 1}};
    static const int kTerms3[6][2] = {{2, 0}, {0, 2}, {1, 1}, {1, 0}, {0, 1}, {0, 0}};      // small terms first
    const int nterm = L.planes == 1 ? 1 : (L.planes == 2 ? 3 : 6);
    p->num_segs = 0;
    p->b_kb_per_tap = L.kb_tap * L.planes;
    p->mma_terms = nterm;
    int kb0 = 0;
    for (int i = 0; i < d.nseg; ++i) {
        if (d.seg[i].cols != L.segc[i]) return fail(h, TMAE_EINVAL, "segment %d width %d != packed %d", i, d.seg[i].cols, L.segc[i]);
        const long long stride = d.seg[i].lo > 0 ? d.seg[i].lo : -d.seg[i].lo;
        const int have = d.seg[i].lo == 0 ? 1 : (d.seg[i].lo > 0 ? 2 : 3);
        if (have != L.planes) return fail(h, TMAE_EINVAL, "layer with %d planes: segment %d has %d", L.planes, i, have);
        const int skb = pad64(d.seg[i].cols) / 64;
        for (int term = 0; term < nterm; ++term) {
            const int pa = L.planes == 3 ? kTerms3[term][0] : (L.planes == 2 ? kTerms2[term][0] : 0);
            const int pw = L.planes == 3 ? kTerms3[term][1] : (L.planes == 2 ? kTerms2[term][1] : 0);
            const int j = p->num_segs++;
            if (j >= kMaxSegs) return fail(h, TMAE_EINVAL, "too many K segments");
            const __nv_bfloat16* ptr = d.seg[i].ptr + pa * stride;
            p->a_ptr[j] = ptr;
            p->a_ld[j] = d.seg[i].ld;
            p->a_cols[j] = d.seg[i].cols;
            p->a_rows[j] = d.a_rows;
            p->seg_kblocks[j] = skb;
            p->seg_b_kb0[j] = kb0 + pw * L.kb_tap;
            int rc = conv ? make_map4d(h, &p->a_map[j], ptr, (uint64_t)d.seg[i].cols, d.side, d.n_img, (uint64_t)d.seg[i].ld, cg.box_n,
                                       cg.box_y + (d.conv_reuse ? 2 : 0))
                          : make_map(h, &p->a_map[j], ptr, (uint64_t)d.seg[i].cols, (uint64_t)d.a_rows, (uint64_t)d.seg[i].ld, kBlockM);
            if (rc) return rc;
        }
        kb0 += skb;
    }
    p->b_ptr = L.w;
    p->b_ld = L.Kp;
    p->num_taps = L.taps;
    p->s = d.side;
    p->K = d.side * d.side;
    p->T = p->K + 1;
    p->n_img = d.n_img; p->box_y = cg.box_y; p->box_n = cg.box_n; p->y_tiles = cg.y_tiles; p->rows_used = cg.rows_used;
    if (d.conv_reuse && !(conv && cg.reuse_ok)) return fail(h, TMAE_EINVAL, "conv_reuse requested for an incompatible tile geometry");
    p->conv_reuse = d.conv_reuse ? 1 : 0;
    p->a_halo_rows = conv ? (cg.box_y + 2) * cg.box_n * d.side : 0;
    p->M = d.M;
    p->N = L.Cout;
    const int m_tiles = (d.M + kBlockM - 1) / kBlockM;
    p->block_n = force_block_n > 0 ? force_block_n : pick_block_n(m_tiles, L.Cout, groups_for_tiling);
    int rc = make_map(h, &p->b_map, L.w, (uint64_t)L.Kp, (uint64_t)L.Cout, (uint64_t)L.Kp, (uint32_t)p->block_n);
    if (rc) return rc;
    p->pair_ok = 0;
    if ((p->block_n & 15) == 0) {                        // CTA-pair launches stage half of the weight tile per CTA
        rc = make_map(h, &p->b_map_pair, L.w, (uint64_t)L.Kp, (uint64_t)L.Cout, (uint64_t)L.Kp, (uint32_t)(p->block_n / 2));
        if (rc) return rc;
        p->pair_ok = 1;
    }
    p->in_mode = d.in_mode;
    // TMA-store epilogue: one bf16 output at the accumulator's own rows, and those rows are 128 consecutive output rows
    {
        const bool one_bf16 = d.out0.dtype == OUT_BF16 && d.out0.map == MAP_SAME && d.out1.dtype == OUT_NONE && d.resid == nullptr &&
                              d.out0.lo_off == 0;        // two-plane outputs take the register store phase
        const bool rows_ok = true;        // conv tiles are stored as the 4-D box they are (any geometry)
        const bool align_ok = (reinterpret_cast<uintptr_t>(d.out0.ptr) & 15) == 0 && ((size_t)d.out0.ld * 2) % 16 == 0;
        p->tma_store_ok = 0;
        if (one_bf16 && rows_ok && align_ok && L.Cout >= 32) {
            const uint64_t out_rows = conv ? (uint64_t)d.a_rows : (uint64_t)d.M;
            int rc2 = conv ? make_map4d(h, &p->out_map, d.out0.ptr, (uint64_t)L.Cout, d.side, d.n_img, (uint64_t)d.out0.ld, cg.box_n, cg.box_y,
                                        32, CU_TENSOR_MAP_SWIZZLE_64B)
                           : make_store_map(h, &p->out_map, d.out0.ptr, (uint64_t)L.Cout, out_rows, (uint64_t)d.out0.ld);
            if (rc2) return rc2;
            p->tma_store_ok = 1;
        }
    }
    p->bias = L.bias;
    p->act = d.act;
    p->resid = d.resid; p->resid_ld = d.resid_ld; p->resid_map = d.resid_map;
    p->gather_ids = d.gather_ids;
    if ((d.ln_stats_in != nullptr) != (L.wsum != nullptr)) return fail(h, TMAE_EINVAL, "LayerNorm fold: layer pack and plan disagree");
    p->ln_stats_in = d.ln_stats_in; p->ln_wsum = L.wsum; p->ln_inv_c = 1.0f / (float)L.Cin; p->ln_eps = h->cfg.ln_eps;
    p->ln_chunks = L.Cin / 32;
    if (d.ln_stats_out != nullptr && L.Cout % 32 != 0) return fail(h, TMAE_EINVAL, "LayerNorm statistics need Cout %% 32 == 0");
    p->ln_stats_out = d.ln_stats_out; p->xbf_out = d.xbf_out;
    p->out[0] = d.out0;
    p->out[1] = d.out1;
    p->flops = d.flops;
    if (d.gc_slice >= 0) {
        const Workspace& w = h->ws;
        if (L.Cout != 2 * h->sc || p->block_n != 32 || (L.Cout & 31) != 0 || L.planes != 1)
            return fail(h, TMAE_EINVAL, "fused Gaussian layer: needs 32-column tiles of a %d-column layer (block_n %d)", L.Cout, p->block_n);
        p->gc_on = d.gc_decode ? 2 : 1;
        p->gc_col0 = d.gc_slice * h->sc;
        p->gc_ld = h->Cy;
        p->gc_pixels = h->K;
        p->gc_y = w.y; p->gc_mu = w.mu; p->gc_sigma = w.sigma; p->gc_yhat = w.yhat;
        p->gc_yhat_bf = w.yhat_bf.p; p->gc_yhat_lo = w.yhat_bf.lo;
        p->gc_rate = w.rate_acc;
        p->gc_table = h->scale_table; p->gc_ntable = h->n_scale_table;
        p->gc_io = w.io;
    }
    return TMAE_OK;
}

// ---- workspace -----------------------------------------------------------------------------------------
// Discards the plans (and their captured graphs) that read any of the DEP_* bits in `mask`.
void drop_plans(tmae_handle* h, unsigned mask) {
    for (auto it = h->plans.begin(); it != h->plans.end();)
        it = (it->second->deps & mask) ? h->plans.erase(it) : std::next(it);
}

void free_pool(std::vector<void*>& pool) {
    for (void* p : pool) cudaFree(p);
    pool.clear();
}

int ensure_workspace(tmae_handle* h, int N) {
    Workspace& w = h->ws;
    if (N <= w.cap_N) return TMAE_OK;
    drop_plans(h, DEP_WS);
    free_pool(w.allocs);
    w = Workspace();
    size_t tot = 0;
    const size_t rt = (size_t)N * h->T, rk = (size_t)N * h->K, rz = (size_t)N * h->s4 * h->s4;
    const size_t rp = rk, rp2 = (size_t)N * h->s2 * h->s2, rp4 = rz;      // every activation is compact: no halo rows
    const int C = h->C, Cy = h->Cy, Cz = h->Cz;
    int ci[5], co[5], aux[5];
#define WS_ALLOC(field, count)                                                        \
    do { int _rc = dev_alloc(h, w.allocs, &(field), (count), &tot); if (_rc) return _rc; } while (0)
    // bf16 activation: one plane, or two (hi, lo) when the layers that read it run split-bf16 (precise)
#define WS_ALLOC_BF(field, count, two)                                                \
    do { const size_t _c = ((size_t)(count) + 63) / 64 * 64;                          \
         const int _pl = (two) ? h->planes : 1;                                       \
         int _rc = dev_alloc(h, w.allocs, &(field).p, _c * _pl, &tot); if (_rc) return _rc; \
         (field).lo = _pl == 1 ? 0 : (_pl == 2 ? (long long)_c : -(long long)_c); } while (0)
    const bool pe = h->precise_enc, pr = h->precise_rate;
    WS_ALLOC(w.ids_keep, rk);
    WS_ALLOC_BF(w.patches, rk * h->patch_dim, pe);
    WS_ALLOC(w.x, rt * C);
    WS_ALLOC_BF(w.xn, rt * C, pe);
    WS_ALLOC_BF(w.x_bf, rt * C, false);
    WS_ALLOC(w.ln_stats, (size_t)2 * h->cfg.encoder_depth * rt * (C / 32) * 2);
    WS_ALLOC_BF(w.qkv, rt * 3 * C, pe);
    WS_ALLOC_BF(w.attn, rt * C, pe);
    WS_ALLOC_BF(w.h1, rt * h->mlp, pe);
    WS_ALLOC_BF(w.enc, rk * C, pr);
    WS_ALLOC_BF(w.ga1, rk * h->ga_ch[1], pr);
    WS_ALLOC_BF(w.ga2, rk * h->ga_ch[2], pr);
    WS_ALLOC_BF(w.ga3, rk * h->ga_ch[3], pr);
    WS_ALLOC_BF(w.y_bf, rp * Cy, pr);
    WS_ALLOC(w.y, rk * Cy);
    WS_ALLOC(w.z, rz * Cz);
    WS_ALLOC(w.mu, rk * Cy);
    WS_ALLOC(w.sigma, rk * Cy);
    WS_ALLOC(w.yhat, rk * Cy);
    WS_ALLOC(w.yhat_force, rk * Cy);
    ha_layers(h, ci, co, aux);
    WS_ALLOC_BF(w.ha1, rp * co[0], pr);
    WS_ALLOC_BF(w.ha2, rp * co[1], pr);
    WS_ALLOC_BF(w.ha3, rp2 * co[2], pr);
    WS_ALLOC_BF(w.ha4, rp2 * co[3], pr);
    WS_ALLOC_BF(w.zhat_bf, rp4 * Cz, pr);
    hs_layers(h, ci, co, aux);
    for (int net = 0; net < 2; ++net) {
        WS_ALLOC_BF(w.hs1[net], rp4 * co[0], pr);
        WS_ALLOC_BF(w.hs2[net], rp2 * co[1], pr);
        WS_ALLOC_BF(w.hs3[net], rp2 * co[2], pr);
        WS_ALLOC_BF(w.hs4[net], rp * co[3], pr);
        WS_ALLOC_BF(w.lat[net], rp * Cy, pr);
    }
    WS_ALLOC_BF(w.yhat_bf, rp * Cy, pr);
    int ch[6];
    cc_channels(h, ch, 0, false);
    for (int net = 0; net < 18; ++net)
        for (int l = 0; l < 4; ++l) WS_ALLOC_BF(w.t[net][l], rp * ch[l + 1], pr);
    WS_ALLOC(w.rate_acc, (size_t)N);
    WS_ALLOC(w.bpp, (size_t)N);
    WS_ALLOC(w.rate_sums, (size_t)2);
    WS_ALLOC(w.st_imgs, (size_t)N * h->cfg.in_chans * h->cfg.img_size * h->cfg.img_size);
    WS_ALLOC(w.st_scores, (size_t)N * h->L);
    WS_ALLOC(w.st_ylik, rk * Cy);
    WS_ALLOC(w.st_zlik, rz * Cz);
    WS_ALLOC(w.st_ysym, rk * Cy);
    WS_ALLOC(w.st_zsym, rz * Cz);
    WS_ALLOC(w.st_ids_restore, (size_t)N * h->L);
    WS_ALLOC(w.io, (size_t)1);
#undef WS_ALLOC_BF
#undef WS_ALLOC
    w.cap_N = N;
    w.bytes = tot;
    return TMAE_OK;
}

size_t workspace_bytes_estimate(const tmae_handle* h, int N) {
    const size_t rt = (size_t)N * h->T, rk = (size_t)N * h->K, rp = rk, rp2 = (size_t)N * h->s2 * h->s2,
                 rp4 = (size_t)N * h->s4 * h->s4;
    const size_t C = h->C;
    size_t b = rk * 8 + rk * h->patch_dim * 2 + rt * C * 4 + rt * C * 2 * 2 + rt * 3 * C * 2 + rt * h->mlp * 2 + rk * C * 2;
    b += rk * (h->ga_ch[1] + h->ga_ch[2] + h->ga_ch[3]) * 2 + rp * h->Cy * 2 + rk * h->Cy * 4 * 4 + rk / 16 * h->Cz * 4;
    b += rp * (384 + 336) * 2 + rp2 * (288 + 240) * 2 + rp4 * h->Cz * 2;
    b += 2 * (rp4 * 240 + rp2 * (288 + 336) + rp * (384 + 384)) * 2 + rp * h->Cy * 2;
    b += 18 * rp * (224 + 176 + 128 + 80) * 2;
    if (h->precise_rate) b += b / 2;            // second bf16 plane of the activations (upper bound)
    if (h->precise_enc) b += b / 3;
    b += (size_t)N * h->cfg.in_chans * h->cfg.img_size * h->cfg.img_size * 4 + (size_t)N * h->L * 4;
    if (h->syn_depth > 0) {          // synthesis buffers (ensure_synth_workspace)
        const size_t sk = (size_t)N * h->K, st = (size_t)N * (h->L + 1), Dd = h->Dd;
        b += sk * (h->Cy + h->ga_ch[3] + h->ga_ch[2] + h->ga_ch[1] + h->C) * 2 + sk * Dd * 4;
        b += st * Dd * (4 + 2 + 3 * 2 + 2) + st * h->syn_mlp * 2 + st * h->syn_out * 2;
        b += (size_t)(2 * h->syn_depth + 1) * st * (Dd / 32) * 8;
    }
    return b;
}

// ---- plan ----------------------------------------------------------------------------------------------
double conv_flops(long long out_positions, int cin, int cout, int taps) {
    return 2.0 * (double)out_positions * cin * cout * taps;
}

// conv_reuse decision for one launch: the geometry must allow it and at least two stages (one haloed A box + three B
// atoms each) must fit the launch's shared-memory budget.  Returns the stage size in bytes, 0 = per-tap loads.
int conv_reuse_stage_bytes(const tmae_handle* h, const GemmDesc& d, int bn, int n_tiles, int groups, bool pair = false) {
    if (d.in_mode != IN_CONV) return 0;
    ConvGeom cg;
    if (!conv_geom(d.side, d.n_img, &cg) || !cg.reuse_ok) return 0;
    const int bn_cta = pair ? bn / 2 : bn;             // B rows this CTA stages (a pair splits the weight tile)
    // a tap's MMA always reads 128 rows from its dy offset: with a partial tile the rows past the A box must still lie
    // inside the stage (they land in the B atoms; the accumulator rows they feed are never stored)
    if (cg.rows_used + 3 * bn_cta < kBlockM) return 0;
    const int stage = ((cg.box_y + 2) * cg.box_n * d.side + 3 * bn_cta) * kBlockK * 2;
    int smem = 0;
    const bool share = (h->cfg.flags & TMAE_FLAG_SHARE_SM) != 0;
    return gemm_reuse_stages(stage, cg.m_tiles * n_tiles * groups, share, &smem) >= 2 ? stage : 0;
}

int add_gemm_group(tmae_handle* h, Plan& pl, const GemmDesc* descs, int groups, const char* tag) {
    Step st;
    st.kind = ST_GEMM;
    st.family = FAM_GEMM;
    st.param_index = (int)pl.host_params.size();
    st.groups = groups;
    st.tag = tag;
    int max_M = 0, max_N = 0;
    for (int g = 0; g < groups; ++g) {
        if (descs[g].M > max_M) max_M = descs[g].M;
        if (descs[g].layer->Cout > max_N) max_N = descs[g].layer->Cout;
    }
    const int m_tiles = (max_M + kBlockM - 1) / kBlockM;
    int bn = pick_block_n(m_tiles, max_N, groups);
    if (descs[0].gc_slice >= 0) bn = 32;        // fused Gaussian epilogue: one 32-column chunk (16 channels: mu | sigma) per CTA
    if (!(h->cfg.flags & TMAE_FLAG_SHARE_SM) && groups == 1 && m_tiles * ((max_N + 255) / 256) > 2 * 148 - 1 && descs[0].out0.dtype == OUT_BF16 && descs[0].out0.map == MAP_SAME &&
        descs[0].out1.dtype == OUT_NONE && descs[0].resid == nullptr) {
        // persistent-kernel candidate: tiles are dealt round-robin to 148 CTAs -> minimise rounds x (tile width + fixed cost)
        long long best_cost = -1;
        for (int cand = 256; cand >= 128; cand -= 16) {
            const int tiles = m_tiles * ((max_N + cand - 1) / cand);
            const long long cost = (long long)((tiles + 147) / 148) * (cand + 48);
            if (best_cost < 0 || cost < best_cost) { best_cost = cost; bn = cand; }
        }
    }
    {   // layers whose store phase can go through TMA (one bf16 same-row output): 32-column boxes -> block_n % 32 == 0
        bool all_bf16_same = !getenv("TMAE_NO_TMA_STORE");
        for (int g = 0; g < groups; ++g)
            all_bf16_same = all_bf16_same && descs[g].out0.dtype == OUT_BF16 && descs[g].out0.map == MAP_SAME &&
                            descs[g].out1.dtype == OUT_NONE && descs[g].resid == nullptr && descs[g].act != ACT_HALF_TANH;
        // conv layers keep their exact tile width (rounding 112 -> 128 or 80 -> 96 computes 14-20 % dead columns; such layers
        // use the register/smem store phase instead): measured equal or slightly better at the power cap
        static const int round_mode = getenv("TMAE_BN_ROUND") ? atoi(getenv("TMAE_BN_ROUND")) : 2;   // 0 never, 1 always, 2 only linear layers
        const bool conv_layer = descs[0].in_mode == IN_CONV;
        if (all_bf16_same && bn % 32 != 0 && bn + 16 <= 256 && (round_mode == 1 || (round_mode == 2 && !conv_layer))) bn += 16;
    }
    for (int g = 0; g < groups; ++g)       // PixelShuffle epilogue: a 32-column chunk must not straddle a quadrant;
        if (descs[g].out0.map == MAP_SHUF || descs[g].out1.map == MAP_SHUF || descs[g].ln_stats_out != nullptr)
            bn = (bn + 31) / 32 * 32;      // LayerNorm statistics: one slot per 32-column chunk, owned by exactly one tile
    // CTA-pair launch?  (decided before the stage sizes: a pair stages half of the weight tile per CTA)
    {
        const bool conv_l = descs[0].in_mode == IN_CONV;
        bool one_bf16 = descs[0].out0.dtype == OUT_BF16 && descs[0].out0.map == MAP_SAME && descs[0].out1.dtype == OUT_NONE && descs[0].resid == nullptr;
        bool f32_resid = descs[0].out0.dtype == OUT_F32 && descs[0].out0.map == MAP_SAME && descs[0].out1.dtype == OUT_NONE &&
                         descs[0].resid != nullptr && descs[0].resid_map == MAP_SAME && descs[0].act == ACT_NONE;
        const int epi_hint = one_bf16 ? 1 : (f32_resid ? 2 : 0);
        st.pair = !(h->cfg.flags & TMAE_FLAG_DEBUG_SIMT) && (bn & 15) == 0 &&
                  gemm_use_pair(groups, epi_hint, descs[0].act, max_M, bn, true, conv_l);
        for (int g = 1; g < groups; ++g) if (descs[g].in_mode != descs[0].in_mode) st.pair = false;
        if (descs[0].gc_slice >= 0) st.pair = false;          // the Gaussian epilogue lives in the one-CTA kernel
    }
    // 3x3 conv launches: haloed-box A reuse when every member agrees on the geometry and the stages fit
    st.conv_reuse_stage_bytes = conv_reuse_stage_bytes(h, descs[0], bn, (max_N + bn - 1) / bn, groups, st.pair);
    for (int g = 1; g < groups; ++g)
        if (descs[g].in_mode != descs[0].in_mode || descs[g].side != descs[0].side || descs[g].n_img != descs[0].n_img) st.conv_reuse_stage_bytes = 0;
    for (int g = 0; g < groups; ++g) {
        GemmParams p;
        GemmDesc dg = descs[g];
        dg.conv_reuse = st.conv_reuse_stage_bytes > 0;
        int rc = fill_params(h, dg, groups, &p, bn);
        if (rc) return rc;
        const int ek = gemm_epi_kind(p);
        if (g == 0) st.epi = ek;
        else if (ek != st.epi) st.epi = ((ek == 1 || ek == 3) && (st.epi == 1 || st.epi == 3)) ? 1 : 0;   // mixed group -> common denominator
        pl.host_params.push_back(p);
        st.flops += descs[g].flops;
        st.mma_terms = p.mma_terms;
    }
    if (descs[0].ln_stats_in != nullptr && st.epi != 3 /*EPI_BF16_TMA*/)
        return fail(h, TMAE_EINVAL, "%s: a LayerNorm-folded layer needs the TMA-store epilogue (epi %d)", tag, st.epi);
    if (descs[0].ln_stats_out != nullptr && st.epi != 2 /*EPI_F32_SAME_RESID*/)
        return fail(h, TMAE_EINVAL, "%s: LayerNorm statistics need the fp32 residual epilogue (epi %d)", tag, st.epi);
    st.max_M = max_M; st.max_N = max_N; st.block_n = bn; st.act = descs[0].act;
    if (st.pair && !pl.host_params[st.param_index].pair_ok) st.pair = false;
    st.pair_persist = st.pair && gemm_use_pair_persistent(groups, st.epi, st.act, max_M, max_N, bn, (h->cfg.flags & TMAE_FLAG_SHARE_SM) != 0,
                                                          descs[0].in_mode == IN_CONV);
    static const bool plan_debug = getenv("TMAE_PLAN_DEBUG") != nullptr;
    if (plan_debug)
        fprintf(stderr, "[plan] %-14s groups %2d M %6d N %4d bn %3d ctas %4d epi %d conv_reuse_stage %6d B pair %d\n", tag, groups, max_M, max_N, bn,
                m_tiles * ((max_N + bn - 1) / bn) * groups, st.epi, st.conv_reuse_stage_bytes, (int)st.pair);
    for (int g = 1; g < groups; ++g) if (descs[g].act != descs[0].act) return fail(h, TMAE_EINVAL, "grouped GEMM members must share the activation");
    pl.steps.push_back(st);
    return TMAE_OK;
}

// Tensor maps of the tcgen05 attention kernel: Q and K / V tiles of one (image, head) are 64-column boxes of qkv [rows, 3C]
int make_attention_maps(tmae_handle* h, const __nv_bfloat16* qkv, long long rows, int C, int T, int mode, CUtensorMap* mq, CUtensorMap* mkv) {
    int q_rows = 0, kv_rows = 0;
    attention_tc_boxes(T, C / 64, mode, &q_rows, &kv_rows);
    cuuint64_t gdim[2] = {(cuuint64_t)(3 * C), (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)(3 * C) * 2};
    cuuint32_t estr[2] = {1, 1};
    cuuint32_t box_q[2] = {64, (cuuint32_t)q_rows}, box_k[2] = {64, (cuuint32_t)kv_rows};
    void* base = const_cast<__nv_bfloat16*>(qkv);
    CUresult r1 = h->encode(mq, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstr, box_q, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult r2 = h->encode(mkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstr, box_k, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS)
        return fail(h, TMAE_ECUDA, "cuTensorMapEncodeTiled(attention) failed (%d %d)", (int)r1, (int)r2);
    return TMAE_OK;
}

SegSrc seg(const __nv_bfloat16* p, int cols, int ld, long long lo = 0) { SegSrc s; s.ptr = p; s.cols = cols; s.ld = ld; s.lo = lo; return s; }
SegSrc seg(const Bf& b, int cols, int ld, int col0 = 0) { return seg(b.p + col0, cols, ld, b.lo); }
OutSpec outspec(void* p, int ld, int dtype, int map, long long lo = 0) { OutSpec o; o.ptr = p; o.ld = ld; o.dtype = dtype; o.map = map; o.lo_off = lo; return o; }
OutSpec outspec(const Bf& b, int ld, int map, int col0 = 0) { return outspec(b.p + col0, ld, OUT_BF16, map, b.lo); }

const Layer* get_layer(tmae_handle* h, const std::string& key) {
    auto it = h->layers.find(key);
    return it == h->layers.end() ? nullptr : &it->second;
}

// 3x3 conv input over a `side` x `side` grid of all N images (compact rows; the tile grid covers box_y x box_n blocks)
void conv_input(GemmDesc& d, int side, int N) {
    ConvGeom cg;
    conv_geom(side, N, &cg);
    d.in_mode = IN_CONV; d.side = side; d.n_img = N;
    d.a_rows = (long long)N * side * side; d.M = cg.m_tiles * kBlockM;
}

// Pieces of the rate half shared by the forward plan (build_plan) and the decode plan (build_decode_plan): the same
// layers with the same launch shapes, so that a decoder reproduces the encoder's mu / sigma / y_hat bit for bit.
// h_s_mean / h_s_scale as a group of two per layer (MCM.py:132-162, 747-748)
int add_hs_steps(tmae_handle* h, Plan& pl, int N) {
    Workspace& w = h->ws;
    const int s = h->s;
    char tag[96];
    int rc;
    auto conv_in = [&](GemmDesc& d, int side) { conv_input(d, side, N); };
    int ci[5], co[5], up[5];
    hs_layers(h, ci, co, up);
    const int sides[5] = {h->s4, h->s4, h->s2, h->s2, s};
    const char* nets[2] = {"h_s_mean", "h_s_scale"};
    for (int l = 0; l < 5; ++l) {
        GemmDesc d[2];
        for (int net = 0; net < 2; ++net) {
            const Bf srcs[5] = {w.zhat_bf, w.hs1[net], w.hs2[net], w.hs3[net], w.hs4[net]};
            const Bf dsts[5] = {w.hs1[net], w.hs2[net], w.hs3[net], w.hs4[net], w.lat[net]};
            d[net].layer = get_layer(h, std::string(nets[net]) + "." + std::to_string(2 * l));
            d[net].seg[0] = seg(srcs[l], ci[l], ci[l]);
            conv_in(d[net], sides[l]);
            d[net].act = l < 4 ? ACT_GELU : ACT_NONE;
            d[net].out0 = outspec(dsts[l], co[l], up[l] == 2 ? MAP_SHUF : MAP_SAME);
            d[net].flops = conv_flops((long long)N * sides[l] * sides[l], ci[l], co[l] * up[l] * up[l], 9);
        }
        snprintf(tag, sizeof(tag), "h_s.%d", 2 * l);
        rc = add_gemm_group(h, pl, d, 2, tag); if (rc) return rc;
    }
    return TMAE_OK;
}

// cc_transform_mean[i] / cc_transform_scale[i] of the slice group [i0, i0 + cnt) (MCM.py:756-768).  decode: the fused last
// layer stores mu, sigma and the scale-table indexes (EPI_GAUSS_IDX) instead of running the Gaussian conditional.
int add_cc_steps(tmae_handle* h, Plan& pl, int N, int i0, int cnt, bool decode) {
    Workspace& w = h->ws;
    const int s = h->s, Cy = h->Cy;
    const long long rk = (long long)N * h->K;
    const int half_sl = h->nsl / 2;
    const int sup = i0 < half_sl ? i0 : half_sl;
    char tag[96];
    int rc;
    auto conv_in = [&](GemmDesc& d, int side) { conv_input(d, side, N); };
    int ch[6];
    cc_channels(h, ch, i0, false);
    for (int l = 0; l < 5; ++l) {    // cc_transform_mean[i] and cc_transform_scale[i] of every member, grouped
        if (l == 4 && h->gc_fuse) {
            // last layers of both nets as ONE block-diagonal GEMM per member (K segments = the two nets' activations);
            // its epilogue is the Gaussian conditional of the slice (MCM.py:762-776): no mu / sigma round trip, no extra launch
            std::vector<GemmDesc> d((size_t)cnt);
            for (int j = 0; j < cnt; ++j) {
                GemmDesc& g = d[(size_t)j];
                const int i = i0 + j;
                g.layer = get_layer(h, "gc." + std::to_string(i));
                g.seg[0] = seg(w.t[j * 3 + 0][3], ch[4], ch[4]);
                g.seg[1] = seg(w.t[j * 3 + 1][3], ch[4], ch[4]);
                g.nseg = 2;
                conv_in(g, s);
                g.gc_slice = i;
                g.gc_decode = decode;
                g.flops = 2.0 * conv_flops(rk, ch[4], ch[5], 9);      // the two layers as the reference counts them (the zero blocks are not work)
            }
            snprintf(tag, sizeof(tag), decode ? "cc.%d.8+idx" : "cc.%d.8+gauss", i0);
            rc = add_gemm_group(h, pl, d.data(), cnt, tag); if (rc) return rc;
            continue;
        }
        std::vector<GemmDesc> d((size_t)cnt * 2);
        for (int j = 0; j < cnt; ++j)
            for (int net = 0; net < 2; ++net) {
                GemmDesc& g = d[(size_t)j * 2 + net];
                const int i = i0 + j;
                const char* nm = net == 0 ? "cc_transform_mean." : "cc_transform_scale.";
                g.layer = get_layer(h, std::string(nm) + std::to_string(i) + "." + std::to_string(2 * l));
                if (l == 0) {
                    g.seg[0] = seg(w.lat[net], Cy, Cy);
                    g.nseg = 1;
                    if (sup > 0) { g.seg[1] = seg(w.yhat_bf, h->sc * sup, Cy); g.nseg = 2; }
                } else {
                    g.seg[0] = seg(w.t[j * 3 + net][l - 1], ch[l], ch[l]);
                }
                conv_in(g, s);
                if (l < 4) { g.act = ACT_GELU; g.out0 = outspec(w.t[j * 3 + net][l], ch[l + 1], MAP_SAME); }
                else g.out0 = outspec((net == 0 ? w.mu : w.sigma) + i * h->sc, Cy, OUT_F32, MAP_SAME);
                g.flops = conv_flops(rk, ch[l], ch[l + 1], 9);
            }
        snprintf(tag, sizeof(tag), "cc.%d.%d", i0, 2 * l);
        rc = add_gemm_group(h, pl, d.data(), cnt * 2, tag); if (rc) return rc;
    }
    return TMAE_OK;
}

// lrp_transform[i] of the slice group (MCM.py:780-783): y_hat += 0.5 tanh(lrp(...)) in place on w.yhat
int add_lrp_steps(tmae_handle* h, Plan& pl, int N, int i0, int cnt, bool forced) {
    Workspace& w = h->ws;
    const int s = h->s, Cy = h->Cy;
    const long long rk = (long long)N * h->K;
    const int half_sl = h->nsl / 2;
    const int sup = i0 < half_sl ? i0 : half_sl;
    char tag[96];
    int rc;
    auto conv_in = [&](GemmDesc& d, int side) { conv_input(d, side, N); };
    int lch[6];
    cc_channels(h, lch, i0, true);
    for (int l = 0; l < 5; ++l) {    // lrp_transform[i] (MCM.py:780-783)
        std::vector<GemmDesc> d((size_t)cnt);
        for (int j = 0; j < cnt; ++j) {
            GemmDesc& g = d[j];
            const int i = i0 + j;
            g.layer = get_layer(h, "lrp_transform." + std::to_string(i) + "." + std::to_string(2 * l));
            if (l == 0) {
                g.seg[0] = seg(w.lat[0], Cy, Cy);
                if (i < half_sl) { g.seg[1] = seg(w.yhat_bf, h->sc * (i + 1), Cy); g.nseg = 2; }
                else { g.seg[1] = seg(w.yhat_bf, h->sc * sup, Cy); g.seg[2] = seg(w.yhat_bf, h->sc, Cy, i * h->sc); g.nseg = 3; }
            } else {
                g.seg[0] = seg(w.t[j * 3 + 2][l - 1], lch[l], lch[l]);
            }
            conv_in(g, s);
            if (l < 4) { g.act = ACT_GELU; g.out0 = outspec(w.t[j * 3 + 2][l], lch[l + 1], MAP_SAME); }
            else {
                g.act = ACT_HALF_TANH;
                g.resid = w.yhat + i * h->sc; g.resid_ld = Cy; g.resid_map = MAP_SAME;
                g.out0 = outspec(w.yhat + i * h->sc, Cy, OUT_F32, MAP_SAME);
                if (!(forced && i < half_sl)) g.out1 = outspec(w.yhat_bf, Cy, MAP_SAME, i * h->sc);
            }
            g.flops = conv_flops(rk, lch[l], lch[l + 1], 9);
        }
        snprintf(tag, sizeof(tag), "lrp.%d.%d", i0, 2 * l);
        rc = add_gemm_group(h, pl, d.data(), cnt, tag); if (rc) return rc;
    }
    return TMAE_OK;
}

// A step that launches one kernel from the plan's buffers (no GEMM parameter block).
void add_step(Plan& pl, StepKind kind, int family, const std::string& tag, int slice = 0, int gc_slices = 1) {
    Step st;
    st.kind = kind; st.family = family; st.tag = tag; st.slice = slice; st.gc_slices = gc_slices;
    pl.steps.push_back(st);
}

// Common tail of every plan: last stage, sanity check, weight-prefetch chain, parameter blocks to the device.
int finish_plan(tmae_handle* h, Plan& pl) {
    pl.stage_begin.push_back((int)pl.steps.size());
    pl.stage_graph.assign(pl.stage_begin.size() - 1, nullptr);
    pl.stage_calls.assign(pl.stage_begin.size() - 1, 0);
    for (const Step& st : pl.steps)
        if (st.kind == ST_GEMM && pl.host_params[st.param_index].num_segs < 1) return fail(h, TMAE_EINVAL, "bad plan");
    if (!getenv("TMAE_NO_WEIGHT_PREFETCH")) {      // each GEMM step prefetches the weights of the next one (cyclically)
        std::vector<int> gemm_steps;
        for (size_t i = 0; i < pl.steps.size(); ++i) if (pl.steps[i].kind == ST_GEMM) gemm_steps.push_back((int)i);
        for (size_t k = 0; k < gemm_steps.size(); ++k) {
            const Step& nx = pl.steps[gemm_steps[(k + 1) % gemm_steps.size()]];
            pl.steps[gemm_steps[k]].next_index = nx.param_index;
            pl.steps[gemm_steps[k]].next_groups = nx.groups;
        }
    }
    void* dp = nullptr;
    CUDA_TRY(h, cudaMalloc(&dp, pl.host_params.size() * sizeof(GemmParams)));
    pl.d_params = reinterpret_cast<GemmParams*>(dp);
    CUDA_TRY(h, cudaMemcpy(pl.d_params, pl.host_params.data(), pl.host_params.size() * sizeof(GemmParams), cudaMemcpyHostToDevice));
    return TMAE_OK;
}

// Pre-norm ViT blocks (timm 0.4.5 Block, eval): QKV -> attention -> proj (+ residual) -> fc1 (GELU) -> fc2 (+ residual) over
// the fp32 residual stream `x`.  The encoder (build_plan) and the MAE decoder of the synthesis plan (build_synth_plan) use it.
struct BlockSet {
    const char* prefix = nullptr;    // weight names "<prefix>.<i>.attn.qkv" ...
    const char* tag = nullptr;       // step tags "<tag><i>.qkv" ...
    int depth = 0, C = 0, mlp = 0, T = 0, N = 0;
    bool fold = false;               // LayerNorm fold: proj / fc2 emit row statistics + a bf16 copy of x, QKV / fc1 apply them
    bool stats_in = false;           // fold: the statistics for block 0's norm1 arrive with the input rows (else a LayerNorm kernel)
    bool stats_out = false;          // fold: the last fc2 emits statistics as well (slot 2 * depth), for a LayerNorm folded after the blocks
    StepKind attn = ST_ATTN;
    float* x = nullptr;
    Bf xn, x_bf, qkv, attn_out, h1;
    float* ln_stats = nullptr;       // [2 * depth (+ 1)][N * T][C / 32][2]
};

int add_blocks(tmae_handle* h, Plan& pl, const BlockSet& b) {
    const int C = b.C, T = b.T, N = b.N;
    const long long rt = (long long)N * T;
    char tag[96];
    int rc;
    if (!b.fold && b.x != h->ws.x) return fail(h, TMAE_EINVAL, "%s: LayerNorm kernels run on the encoder's buffers only", b.prefix);
    for (int i = 0; i < b.depth; ++i) {
        const std::string pre = std::string(b.prefix) + "." + std::to_string(i);
        // LayerNorm fold: in the encoder, norm1 of block 0 follows the patch embed + cls rows and stays a kernel; every other
        // block LayerNorm lives in the GEMMs around it - proj / fc2 emit row statistics + a bf16 copy of x, QKV / fc1 apply them
        const bool fold1 = b.fold && (i > 0 || b.stats_in), fold2 = b.fold;
        const size_t stat_stride = (size_t)rt * (C / 32) * 2;
        float* stats1 = b.ln_stats + (size_t)(2 * i) * stat_stride;          // statistics of x entering norm1 / norm2 of block i
        float* stats2 = b.ln_stats + (size_t)(2 * i + 1) * stat_stride;
        if (!fold1) {
            Step ln; ln.kind = ST_LN; ln.family = FAM_LN; ln.ln_gamma = h->vecs[pre + ".norm1.weight"]; ln.ln_beta = h->vecs[pre + ".norm1.bias"]; ln.tag = pre + ".norm1";
            pl.steps.push_back(ln);
        }
        GemmDesc d;
        d.layer = get_layer(h, pre + ".attn.qkv");
        d.seg[0] = fold1 ? seg(b.x_bf, C, C) : seg(b.xn, C, C); d.a_rows = rt; d.M = (int)rt;
        if (fold1) d.ln_stats_in = stats1;
        d.out0 = outspec(b.qkv, 3 * C, MAP_SAME);
        d.flops = 2.0 * rt * C * 3.0 * C;
        snprintf(tag, sizeof(tag), "%s%d.qkv", b.tag, i);
        rc = add_gemm_group(h, pl, &d, 1, tag); if (rc) return rc;
        Step at; at.kind = b.attn; at.family = FAM_ATTN; at.flops = 4.0 * (double)N * T * T * C; at.tag = pre + ".attn";
        pl.steps.push_back(at);
        GemmDesc p2;
        p2.layer = get_layer(h, pre + ".attn.proj");
        p2.seg[0] = seg(b.attn_out, C, C); p2.a_rows = rt; p2.M = (int)rt;
        p2.resid = b.x; p2.resid_ld = C; p2.resid_map = MAP_SAME;
        p2.out0 = outspec(b.x, C, OUT_F32, MAP_SAME);
        if (fold2) { p2.ln_stats_out = stats2; p2.xbf_out = b.x_bf.p; }
        p2.flops = 2.0 * rt * C * (double)C;
        snprintf(tag, sizeof(tag), "%s%d.proj", b.tag, i);
        rc = add_gemm_group(h, pl, &p2, 1, tag); if (rc) return rc;
        if (!fold2) {
            Step ln2; ln2.kind = ST_LN; ln2.family = FAM_LN; ln2.ln_gamma = h->vecs[pre + ".norm2.weight"]; ln2.ln_beta = h->vecs[pre + ".norm2.bias"]; ln2.tag = pre + ".norm2";
            pl.steps.push_back(ln2);
        }
        GemmDesc f1;
        f1.layer = get_layer(h, pre + ".mlp.fc1");
        f1.seg[0] = fold2 ? seg(b.x_bf, C, C) : seg(b.xn, C, C); f1.a_rows = rt; f1.M = (int)rt; f1.act = ACT_GELU;
        if (fold2) f1.ln_stats_in = stats2;
        f1.out0 = outspec(b.h1, b.mlp, MAP_SAME);
        f1.flops = 2.0 * rt * C * (double)b.mlp;
        snprintf(tag, sizeof(tag), "%s%d.fc1", b.tag, i);
        rc = add_gemm_group(h, pl, &f1, 1, tag); if (rc) return rc;
        GemmDesc f2;
        f2.layer = get_layer(h, pre + ".mlp.fc2");
        f2.seg[0] = seg(b.h1, b.mlp, b.mlp); f2.a_rows = rt; f2.M = (int)rt;
        f2.resid = b.x; f2.resid_ld = C; f2.resid_map = MAP_SAME;
        f2.out0 = outspec(b.x, C, OUT_F32, MAP_SAME);
        if (b.fold && (i + 1 < b.depth || b.stats_out)) {                    // statistics for norm1 of the next block
            f2.ln_stats_out = b.ln_stats + (size_t)(2 * i + 2) * stat_stride; f2.xbf_out = b.x_bf.p;
        }
        f2.flops = 2.0 * rt * C * (double)b.mlp;
        snprintf(tag, sizeof(tag), "%s%d.fc2", b.tag, i);
        rc = add_gemm_group(h, pl, &f2, 1, tag); if (rc) return rc;
    }
    return TMAE_OK;
}

// forced = slice-wise teacher forcing (tmae_forward_from_latent_forced): after lrp_transform[i] the support columns of
// slice i are overwritten with the caller's y_hat, so slice j > i never sees a symbol this run decided itself.
int build_plan(tmae_handle* h, Plan& pl, bool forced) {
    const int N = pl.N;
    int rc = ensure_workspace(h, N);
    if (rc) return rc;
    Workspace& w = h->ws;
    const int C = h->C, T = h->T, K = h->K, s = h->s, Cy = h->Cy, Cz = h->Cz;
    const long long rt = (long long)N * T, rk = (long long)N * K;
    char tag[96];
    auto conv_in = [&](GemmDesc& d, int side) { conv_input(d, side, N); };

    if (!h->precise_enc && !(h->cfg.flags & TMAE_FLAG_DEBUG_SIMT) && attention_tc_eligible(T)) {
        if ((rc = make_attention_maps(h, w.qkv.p, rt, C, T, (h->cfg.flags & TMAE_FLAG_SHARE_SM) ? 2 : 1, &pl.attn_q, &pl.attn_k))) return rc;
        pl.attn_tc = true;
    }
    add_step(pl, ST_ZERO_RATE, FAM_MISC, "zero_rate");
    add_step(pl, ST_MASK, FAM_MASK, "mask_select");
    add_step(pl, ST_GATHER, FAM_GATHER, "gather_patches");
    {   // patch embed: conv k16 s16 == linear over (c,p,q) patches; + bias + pos_embed[id+1]  (MCM.py:615-618)
        GemmDesc d;
        d.layer = get_layer(h, "encoder_embed.proj");
        d.seg[0] = seg(w.patches, h->patch_dim, h->patch_dim);
        d.a_rows = rk; d.M = (int)rk; d.in_mode = IN_COMPACT; d.side = s;
        d.resid = h->vecs["encoder_pos_embed"]; d.resid_ld = C; d.resid_map = MAP_GATHER1; d.gather_ids = w.ids_keep;
        d.out0 = outspec(w.x, C, OUT_F32, MAP_TO_TOKEN);
        d.flops = 2.0 * (double)rk * h->patch_dim * C;             // executed: the K kept patches (the reference embeds all L: bench adds that figure)
        rc = add_gemm_group(h, pl, &d, 1, "patch_embed");
        if (rc) return rc;
    }
    {
        BlockSet b;
        b.prefix = "encoder_blocks"; b.tag = "blk";
        b.depth = h->cfg.encoder_depth; b.C = C; b.mlp = h->mlp; b.T = T; b.N = N;
        b.fold = h->ln_fold; b.attn = ST_ATTN;
        b.x = w.x; b.xn = w.xn; b.x_bf = w.x_bf; b.qkv = w.qkv; b.attn_out = w.attn; b.h1 = w.h1; b.ln_stats = w.ln_stats;
        if ((rc = add_blocks(h, pl, b))) return rc;
    }
    {
        Step ln; ln.kind = ST_LN; ln.family = FAM_LN; ln.ln_gamma = h->vecs["encoder_norm.weight"]; ln.ln_beta = h->vecs["encoder_norm.bias"]; ln.ln_final = 1; ln.tag = "encoder_norm";
        pl.steps.push_back(ln);
    }
    pl.encoder_end_step = (int)pl.steps.size();
    {   // g_a: four 1x1 convs == per-token linears (MCM.py:77-93, 735)
        const Bf srcs[4] = {w.enc, w.ga1, w.ga2, w.ga3};
        const Bf dsts[3] = {w.ga1, w.ga2, w.ga3};
        for (int l = 0; l < 4; ++l) {
            GemmDesc d;
            d.layer = get_layer(h, "g_a." + std::to_string(2 * l));
            d.seg[0] = seg(srcs[l], h->ga_ch[l], h->ga_ch[l]); d.a_rows = rk; d.M = (int)rk;
            d.in_mode = IN_COMPACT; d.side = s;
            if (l < 3) { d.act = ACT_GELU; d.out0 = outspec(dsts[l], h->ga_ch[l + 1], MAP_SAME); }
            else { d.out0 = outspec(w.y, Cy, OUT_F32, MAP_SAME); d.out1 = outspec(w.y_bf, Cy, MAP_SAME); }
            d.flops = 2.0 * rk * h->ga_ch[l] * (double)h->ga_ch[l + 1];
            snprintf(tag, sizeof(tag), "g_a.%d", 2 * l);
            rc = add_gemm_group(h, pl, &d, 1, tag); if (rc) return rc;
        }
    }
    pl.first_rate_step = (int)pl.steps.size();
    {   // h_a (MCM.py:115-129, 739)
        int ci[5], co[5], st[5];
        ha_layers(h, ci, co, st);
        const Bf srcs[5] = {w.y_bf, w.ha1, w.ha2, w.ha3, w.ha4};
        const Bf dsts[4] = {w.ha1, w.ha2, w.ha3, w.ha4};
        const int sides[5] = {s, s, s, h->s2, h->s2};
        for (int l = 0; l < 5; ++l) {
            GemmDesc d;
            d.layer = get_layer(h, "h_a." + std::to_string(2 * l));
            d.seg[0] = seg(srcs[l], ci[l], ci[l]);
            conv_in(d, sides[l]);
            if (l < 4) { d.act = ACT_GELU; d.out0 = outspec(dsts[l], co[l], st[l] == 2 ? MAP_S2 : MAP_SAME); }
            else d.out0 = outspec(w.z, Cz, OUT_F32, st[l] == 2 ? MAP_S2 : MAP_SAME);
            const long long outpos = (long long)N * (sides[l] / st[l]) * (sides[l] / st[l]);
            d.flops = conv_flops(outpos, ci[l], co[l], 9);
            snprintf(tag, sizeof(tag), "h_a.%d", 2 * l);
            rc = add_gemm_group(h, pl, &d, 1, tag); if (rc) return rc;
        }
    }
    add_step(pl, ST_EB, FAM_ENTROPY, "entropy_bottleneck");
    if ((rc = add_hs_steps(h, pl, N))) return rc;
    const bool skip_dead = (h->cfg.flags & TMAE_FLAG_SKIP_DEAD_LRP) != 0;
    // Slice loop (MCM.py:755-784).  Slice i reads y_hat of slices [0, min(i, 6)): slices 0..5 form a serial chain,
    // slices 6..11 depend only on 0..5 and are mutually independent, so they run as ONE grouped launch per layer.
    const int half_sl = h->nsl / 2;
    for (int i0 = 0; i0 < h->nsl;) {
        const int cnt = i0 < half_sl ? 1 : h->nsl - i0;          // members of this slice group
        if ((rc = add_cc_steps(h, pl, N, i0, cnt, false))) return rc;
        if (!h->gc_fuse) add_step(pl, ST_GC, FAM_ENTROPY, "gaussian." + std::to_string(i0), i0, cnt);
        if (!(skip_dead && i0 >= half_sl) && (rc = add_lrp_steps(h, pl, N, i0, cnt, forced))) return rc;
        if (forced && i0 < half_sl) add_step(pl, ST_FORCE, FAM_MISC, "force." + std::to_string(i0), i0);
        i0 += cnt;
    }
    add_step(pl, ST_RATE, FAM_ENTROPY, "rate_finalize");

    // algorithmic HBM bytes of the memory-bound kernels (bench.py reports them against the measured HBM peak)
    for (Step& st : pl.steps) {
        const double rows_t = (double)N * T, rows_k = (double)N * K, rows_z = (double)N * h->s4 * h->s4;
        switch (st.kind) {
            case ST_LN: st.bytes = st.ln_final ? rows_t * C * 4 + rows_k * C * (2 + 4) : rows_t * C * (4 + 2); break;
            case ST_MASK: st.bytes = (double)N * h->L * (4 + 8 + 8) + rows_k * 8; break;
            case ST_GATHER: st.bytes = rows_k * h->patch_dim * (4 + 2) + (double)N * C * 4; break;
            case ST_EB: st.bytes = rows_z * Cz * (4 + 4 + 4 + 4 + 2); break;
            case ST_GC: st.bytes = rows_k * h->sc * st.gc_slices * (3 * 4 + 3 * 4 + 2); break;
            default: break;
        }
    }
    return TMAE_OK;
}

// Slice groups of the chain (MCM.py:755-784): slices 0 .. nsl/2 - 1 one at a time, then nsl/2 .. nsl - 1 together (they read
// only y_hat of the first half).  The forward plan and the decode stages split the slices the same way.
void slice_groups(int nsl, std::vector<std::pair<int, int>>& g) {
    g.clear();
    const int half_sl = nsl / 2;
    for (int i0 = 0; i0 < nsl;) {
        const int cnt = i0 < half_sl ? 1 : nsl - i0;
        g.push_back({i0, cnt});
        i0 += cnt;
    }
}

int ensure_coder_workspace(tmae_handle* h, int N) {
    CoderWorkspace& c = h->cws;
    if (N <= c.cap_N) return TMAE_OK;
    drop_plans(h, DEP_CODER);
    for (void* p : c.allocs) cudaFree(p);
    c.allocs.clear();
    c.cap_N = 0;
    const size_t ny = (size_t)N * h->Cy * h->K, nz = (size_t)N * h->Cz * h->s4 * h->s4;
    int rc;
    if ((rc = dev_alloc(h, c.allocs, &c.zsym, nz)) || (rc = dev_alloc(h, c.allocs, &c.ysym, ny)) ||
        (rc = dev_alloc(h, c.allocs, &c.idx, ny)) || (rc = dev_alloc(h, c.allocs, &c.state, (size_t)N * 32)))
        return rc;
    c.cap_N = N;
    return TMAE_OK;
}

// Decode plan (MCM.decompress, MCM.py:896-968): the rate half of the forward with y replaced by symbols.
// lrp_transform[6..11] always runs: y_hat is the product here (TMAE_FLAG_SKIP_DEAD_LRP applies to the forward only).
// Uncoded (tmae_decode_begin / _step, the caller's range decoder supplies the symbols): cut into stages at the slice groups,
// because the range decoder needs the scale-table indexes of a group before it can supply the group's symbols.
//   stage 0      z dequantise, h_s, cc layers + indexes of group 0
//   stage g + 1  dequantise group g (symbols + mu), lrp_transform of group g, then cc layers + indexes of group g + 1
//                (after the last group: y_hat / mu / sigma to the caller's buffers)
// Coded (tmae_decompress_streams): the range decoder in front of the two dequantisations - ST_ZDEC decodes the z streams with
// the bottleneck tables before ST_ZDEQ, and ST_YDEC decodes slice group g of the y streams, with the indexes the group's cc
// layers just wrote, before ST_YDEQ.  The y decoder's state stays in the coder workspace between the groups.  One stage: the
// whole decode replays as one CUDA graph per (batch size, lanes).  lanes_y / lanes_z = 0: compressai's format; else the laned
// format with that many lanes per y / z stream.
int build_decode_plan(tmae_handle* h, Plan& pl, bool coded, int lanes_y, int lanes_z) {
    const int N = pl.N;
    int rc = ensure_workspace(h, N);
    if (rc || (coded && (rc = ensure_coder_workspace(h, N)))) return rc;
    std::vector<std::pair<int, int>> groups;
    slice_groups(h->nsl, groups);
    if (coded) {
        add_step(pl, ST_ZDEC, FAM_CODER, "rans_decode.z");
        pl.steps.back().lanes = lanes_z;
    }
    add_step(pl, ST_ZDEQ, FAM_ENTROPY, "z_dequantize");
    if ((rc = add_hs_steps(h, pl, N))) return rc;
    for (const auto& g : groups) {
        if ((rc = add_cc_steps(h, pl, N, g.first, g.second, true))) return rc;
        if (!h->gc_fuse) add_step(pl, ST_IDX, FAM_ENTROPY, "indexes." + std::to_string(g.first), g.first, g.second);
        if (coded) {
            add_step(pl, ST_YDEC, FAM_CODER, "rans_decode.y." + std::to_string(g.first), g.first, g.second);
            pl.steps.back().lanes = lanes_y;
        } else {
            pl.stage_begin.push_back((int)pl.steps.size());
        }
        add_step(pl, ST_YDEQ, FAM_ENTROPY, "dequantize." + std::to_string(g.first), g.first, g.second);
        if ((rc = add_lrp_steps(h, pl, N, g.first, g.second, false))) return rc;
    }
    add_step(pl, ST_DEC_OUT, FAM_MISC, "decode_outputs");
    return TMAE_OK;
}

int ensure_synth_workspace(tmae_handle* h, int N) {
    SynthWorkspace& w = h->sws;
    if (N <= w.cap_N) return TMAE_OK;
    drop_plans(h, DEP_SYNTH);
    free_pool(w.allocs);
    w = SynthWorkspace();
    const size_t rk = (size_t)N * h->K, rt = (size_t)N * (h->L + 1), Dd = h->Dd;
    int rc;
    auto bf = [&](Bf& b, size_t count) { return dev_alloc(h, w.allocs, &b.p, (count + 63) / 64 * 64); };
    if ((rc = bf(w.y_bf, rk * h->Cy)) || (rc = bf(w.gs[0], rk * h->ga_ch[3])) || (rc = bf(w.gs[1], rk * h->ga_ch[2])) ||
        (rc = bf(w.gs[2], rk * h->ga_ch[1])) || (rc = bf(w.tok, rk * h->C)) || (rc = dev_alloc(h, w.allocs, &w.emb, rk * Dd)) ||
        (rc = dev_alloc(h, w.allocs, &w.x, rt * Dd)) || (rc = bf(w.x_bf, rt * Dd)) || (rc = bf(w.qkv, rt * 3 * Dd)) ||
        (rc = bf(w.attn, rt * Dd)) || (rc = bf(w.h1, rt * h->syn_mlp)) || (rc = bf(w.pred, rt * h->syn_out)) ||
        (rc = dev_alloc(h, w.allocs, &w.ln_stats, (size_t)(2 * h->syn_depth + 1) * rt * (Dd / 32) * 2)) ||
        (rc = dev_alloc(h, w.allocs, &w.io, (size_t)1)))
        return rc;
    w.cap_N = N;
    return TMAE_OK;
}

// Synthesis plan (recon.synthesize, MCM.py:789-792 and 636-688, on the engine): x_hat from y_hat and ids_restore.  bf16 operands,
// fp32 accumulation, fp32 residual stream / LayerNorm statistics / softmax, in every accuracy mode (the precise flags govern the
// rate path; no symbol depends on x_hat).  Every LayerNorm is folded: block 0's norm1 into its QKV with the statistics the
// unshuffle writes, decoder_norm into decoder_pred with the statistics of the last fc2.  One stage: one CUDA graph per N.
int build_synth_plan(tmae_handle* h, Plan& pl) {
    const int N = pl.N;
    int rc = ensure_synth_workspace(h, N);
    if (rc) return rc;
    SynthWorkspace& w = h->sws;
    const int Dd = h->Dd, T = h->L + 1, Cy = h->Cy;
    const long long rk = (long long)N * h->K, rt = (long long)N * T;
    add_step(pl, ST_SYN_IN, FAM_MISC, "synth_input");
    {   // g_s: four 1x1 ConvTranspose2d == per-token linears, GELU after the first three (MCM.py:96-112, 790)
        const int ch[5] = {Cy, h->ga_ch[3], h->ga_ch[2], h->ga_ch[1], h->C};
        const Bf srcs[4] = {w.y_bf, w.gs[0], w.gs[1], w.gs[2]}, dsts[4] = {w.gs[0], w.gs[1], w.gs[2], w.tok};
        char tag[32];
        for (int l = 0; l < 4; ++l) {
            GemmDesc d;
            d.layer = get_layer(h, "g_s." + std::to_string(2 * l));
            d.seg[0] = seg(srcs[l], ch[l], ch[l]); d.a_rows = rk; d.M = (int)rk;
            d.act = l < 3 ? ACT_GELU : ACT_NONE;
            d.out0 = outspec(dsts[l], ch[l + 1], MAP_SAME);
            d.flops = 2.0 * rk * ch[l] * (double)ch[l + 1];
            snprintf(tag, sizeof(tag), "g_s.%d", 2 * l);
            if ((rc = add_gemm_group(h, pl, &d, 1, tag))) return rc;
        }
    }
    {   // decoder_embed (MCM.py:638), fp32 out: the unshuffle builds the residual stream from it
        GemmDesc d;
        d.layer = get_layer(h, "decoder_embed");
        d.seg[0] = seg(w.tok, h->C, h->C); d.a_rows = rk; d.M = (int)rk;
        d.out0 = outspec(w.emb, Dd, OUT_F32, MAP_SAME);
        d.flops = 2.0 * rk * h->C * (double)Dd;
        if ((rc = add_gemm_group(h, pl, &d, 1, "decoder_embed"))) return rc;
    }
    add_step(pl, ST_UNSHUF, FAM_GATHER, "unshuffle");
    {
        BlockSet b;
        b.prefix = "decoder_blocks"; b.tag = "dec_blk";
        b.depth = h->syn_depth; b.C = Dd; b.mlp = h->syn_mlp; b.T = T; b.N = N;
        b.fold = true; b.stats_in = true; b.stats_out = true; b.attn = ST_ATTN32;
        b.x = w.x; b.x_bf = w.x_bf; b.qkv = w.qkv; b.attn_out = w.attn; b.h1 = w.h1; b.ln_stats = w.ln_stats;
        if ((rc = add_blocks(h, pl, b))) return rc;
    }
    {   // decoder_norm folded into decoder_pred (MCM.py:684-686); every row, row 0 is dropped by the unpatchify
        GemmDesc d;
        d.layer = get_layer(h, "decoder_pred");
        d.seg[0] = seg(w.x_bf, Dd, Dd); d.a_rows = rt; d.M = (int)rt;
        d.ln_stats_in = w.ln_stats + (size_t)(2 * h->syn_depth) * rt * (Dd / 32) * 2;
        d.out0 = outspec(w.pred, h->syn_out, MAP_SAME);
        d.flops = 2.0 * rt * Dd * (double)h->syn_out;
        if ((rc = add_gemm_group(h, pl, &d, 1, "decoder_pred"))) return rc;
    }
    add_step(pl, ST_UNPATCH, FAM_MISC, "unpatchify");
    for (Step& st : pl.steps) {      // algorithmic HBM bytes of the elementwise steps
        switch (st.kind) {
            case ST_SYN_IN: st.bytes = (double)rk * Cy * (4 + 2); break;
            case ST_UNSHUF: st.bytes = (double)rt * Dd * (4 + 4 + 2) + (double)rt * (Dd / 32) * 8 + (double)N * h->L * 8; break;
            case ST_UNPATCH: st.bytes = (double)N * h->L * h->syn_out * (2 + 4); break;
            default: break;
        }
    }
    return TMAE_OK;
}

// The plan of `kind` for batch size N (lanes: PLAN_STREAMS only), built on first use and kept until drop_plans discards it.
int get_plan(tmae_handle* h, PlanKind kind, int N, Plan** out, int lanes_y = 0, int lanes_z = 0) {
    const PlanKey key(kind, N, lanes_y, lanes_z);
    auto it = h->plans.find(key);
    if (it != h->plans.end()) { *out = it->second.get(); return TMAE_OK; }
    std::unique_ptr<Plan> pl(new Plan());
    pl->N = N;
    pl->deps = kPlanDeps[kind];
    int rc = TMAE_OK;
    switch (kind) {
        case PLAN_FORWARD: case PLAN_FORCED: rc = build_plan(h, *pl, kind == PLAN_FORCED); break;
        case PLAN_DECODE: case PLAN_STREAMS: rc = build_decode_plan(h, *pl, kind == PLAN_STREAMS, lanes_y, lanes_z); break;
        case PLAN_SYNTH: rc = build_synth_plan(h, *pl); break;
    }
    if (rc || (rc = finish_plan(h, *pl))) return rc;
    *out = pl.get();
    h->plans[key] = std::move(pl);
    return TMAE_OK;
}

// ---- execution -----------------------------------------------------------------------------------------
struct RunArgs {
    const float* imgs = nullptr;
    const float* scores = nullptr;
    const tmae_outputs* out = nullptr;
    int begin = 0, end = 0;
    const IoBlock* io = nullptr;     // non-null: kernels read the per-call pointers from the device IoBlock
};

// The next profiling record, started at step `st` with no launches counted yet.
int prof_slot(tmae_handle* h, const Step& st, ProfRecord** out) {
    if (h->prof_used == h->prof.size()) {
        ProfRecord r;
        CUDA_TRY(h, cudaEventCreate(&r.begin));
        CUDA_TRY(h, cudaEventCreate(&r.end));
        h->prof.push_back(r);
    }
    ProfRecord& r = h->prof[h->prof_used++];
    r.family = st.family;
    r.flops = r.bytes = r.mma_flops = 0;
    r.tag = st.tag;
    r.ctas = st.kind == ST_GEMM ? ((st.max_M + kBlockM - 1) / kBlockM) * ((st.max_N + st.block_n - 1) / st.block_n) * st.groups : 0;
    r.block_n = st.kind == ST_GEMM ? st.block_n : 0;
    r.launches = 0;
    *out = &r;
    return TMAE_OK;
}

int run_steps(tmae_handle* h, Plan& pl, const RunArgs& a, cudaStream_t st) {
    Workspace& w = h->ws;
    const int N = pl.N, C = h->C, T = h->T, K = h->K, s = h->s;
    static const tmae_outputs kNoOut = {};
    const tmae_outputs& o = a.out ? *a.out : kNoOut;
    const bool simt = (h->cfg.flags & TMAE_FLAG_DEBUG_SIMT) != 0;
    if (a.io == nullptr && h->gc_fuse) {
        // plain launches: the fused Gaussian epilogue always reads the caller's output pointers from the device IoBlock
        IoBlock hio;
        memset(&hio, 0, sizeof(hio));
        hio.out = o;
        CUDA_TRY(h, cudaMemcpyAsync(w.io, &hio, sizeof(hio), cudaMemcpyHostToDevice, st));   // pageable source: staged before return
    }
    for (int si = a.begin; si < a.end; ++si) {
        const Step& sp = pl.steps[si];
        // profiling: per launch, or (prof_by_run) per run of consecutive launches of one kernel family, which keeps
        // the launch-to-launch overlap inside a run and drops the event gap between its members
        const bool run_start = !h->prof_by_run || si == a.begin || pl.steps[si - 1].family != sp.family;
        const bool run_end = !h->prof_by_run || si + 1 == a.end || pl.steps[si + 1].family != sp.family;
        if (h->profiling) {
            if (run_start) {
                ProfRecord* r = nullptr;
                int rc = prof_slot(h, sp, &r);
                if (rc) return rc;
                CUDA_TRY(h, cudaEventRecord(r->begin, st));
            }
            ProfRecord& r = h->prof[h->prof_used - 1];
            r.flops += sp.flops;
            r.bytes += sp.bytes;
            r.mma_flops += sp.flops * sp.mma_terms;
            r.launches += 1;
        }
        switch (sp.kind) {
            case ST_ZERO_RATE:
                CUDA_TRY(h, cudaMemsetAsync(w.rate_acc, 0, sizeof(double) * N, st));
                break;
            case ST_MASK:
                CUDA_TRY(h, launch_mask_select(a.scores, N, h->L, K, h->cfg.softmax_isa == 8 ? 8 : 16, o.ids_shuffle,
                                               o.ids_restore, w.ids_keep, st, a.io));
                break;
            case ST_GATHER:
                CUDA_TRY(h, launch_gather_patches(a.imgs, w.ids_keep, w.patches.p, w.x, h->vecs["cls_token"],
                                                  h->vecs["encoder_pos_embed"], N, h->cfg.img_size, h->grid_w, K, T, C,
                                                  h->cfg.in_chans, h->cfg.patch_size, w.patches.lo, st, a.io));
                break;
            case ST_GEMM:
                CUDA_TRY(h, gemm_launch(pl.d_params + sp.param_index, sp.groups, sp.max_M, sp.max_N, sp.block_n, sp.act, sp.epi, simt, (h->cfg.flags & TMAE_FLAG_SHARE_SM) != 0, st,
                                        sp.next_index >= 0 ? pl.d_params + sp.next_index : nullptr, sp.next_groups, sp.conv_reuse_stage_bytes, sp.pair ? (sp.pair_persist ? 2 : 1) : 0));
                break;
            case ST_FORCE:
                CUDA_TRY(h, launch_f32_to_bf16_cols(w.yhat_force + sp.slice * h->sc, w.yhat_bf.p + sp.slice * h->sc, (long long)N * K, h->sc,
                                                    h->Cy, w.yhat_bf.lo, st));
                break;
            case ST_LN:
                if (sp.ln_final)
                    CUDA_TRY(h, launch_layernorm(w.x, sp.ln_gamma, sp.ln_beta, w.enc.p, o.x_remain, N * T, C, T, 1, h->cfg.ln_eps, w.enc.lo, st, a.io));
                else
                    CUDA_TRY(h, launch_layernorm(w.x, sp.ln_gamma, sp.ln_beta, w.xn.p, nullptr, N * T, C, T, 0, h->cfg.ln_eps, w.xn.lo, st));
                break;
            case ST_ATTN:
                if (h->precise_enc)
                    CUDA_TRY(h, launch_attention_f32(w.qkv.p, w.qkv.lo, w.attn.p, w.attn.lo, N, T, h->H, C, 1.0f / sqrtf((float)h->hd), st));
                else if (pl.attn_tc)
                    CUDA_TRY(h, launch_attention_tc(&pl.attn_q, &pl.attn_k, w.qkv.p, w.attn.p, N, T, h->H, C, 1.0f / sqrtf((float)h->hd), st, nullptr,
                                                    (h->cfg.flags & TMAE_FLAG_SHARE_SM) ? 2 : 1));
                else
                    CUDA_TRY(h, launch_attention(w.qkv.p, w.attn.p, N, T, h->H, C, 1.0f / sqrtf((float)h->hd), st));
                break;
            case ST_EB:
                CUDA_TRY(h, launch_bottleneck(w.z, h->eb_tab, (long long)N * h->s4 * h->s4, h->Cz, o.z_likelihoods,
                                              o.z_symbols, o.z_hat, w.zhat_bf.p, w.zhat_bf.lo, h->s4, w.rate_acc, h->s4 * h->s4,
                                              o.z_symbols_i16, st, a.io));
                break;
            case ST_GC:
                CUDA_TRY(h, launch_gaussian_slice(w.y, w.mu, w.sigma, (long long)N * K, h->Cy, sp.slice * h->sc, h->sc * sp.gc_slices,
                                                  o.y_likelihoods, o.y_symbols, w.yhat, w.yhat_bf.p, w.yhat_bf.lo, h->Cy, s, w.rate_acc,
                                                  h->scale_table, h->n_scale_table, o.y_symbols_i16, o.y_indexes, st, a.io));
                break;
            case ST_RATE:
                CUDA_TRY(h, launch_rate_finalize(w.rate_acc, N, (double)h->cfg.img_size * h->cfg.img_size,
                                                 o.bpp ? o.bpp : w.bpp, o.rate_sums ? o.rate_sums : w.rate_sums, st, a.io));
                break;
            case ST_ZDEQ:
                CUDA_TRY(h, launch_z_dequantize(h->eb_tab, (long long)N * h->s4 * h->s4, h->Cz, h->s4 * h->s4, w.zhat_bf.p, w.zhat_bf.lo, st, a.io));
                break;
            case ST_IDX:
                CUDA_TRY(h, launch_slice_indexes(w.sigma, (long long)N * K, h->Cy, sp.slice * h->sc, h->sc * sp.gc_slices, K, h->scale_table,
                                                 h->n_scale_table, st, a.io));
                break;
            case ST_YDEQ:
                CUDA_TRY(h, launch_slice_dequantize(w.mu, (long long)N * K, h->Cy, sp.slice * h->sc, h->sc * sp.gc_slices, K, w.yhat, w.yhat_bf.p,
                                                    w.yhat_bf.lo, st, a.io));
                break;
            case ST_DEC_OUT:
                CUDA_TRY(h, launch_copy_outputs(a.io, w.y, w.z, w.mu, w.sigma, w.yhat, w.ids_keep, (long long)N * K * h->Cy,
                                                (long long)N * h->s4 * h->s4 * h->Cz, (long long)N * K, st));
                break;
            case ST_ZDEC: {
                const CdfTables& t = h->cdf[TMAE_MODEL_BOTTLENECK];
                RansDecArgs d;
                d.cdf = t.cdf; d.entries = t.entries; d.n_tab = t.n;
                d.idx_div = h->s4 * h->s4;
                d.symbols = h->cws.zsym; d.sym_stride = (long long)h->Cz * h->s4 * h->s4;
                d.n_streams = N; d.begin = 0; d.end = h->Cz * h->s4 * h->s4;
                d.lanes = sp.lanes;
                d.io = a.io; d.io_stream = 2;
                CUDA_TRY(h, launch_rans_decode(d, st));
                break;
            }
            case ST_SYN_IN:
                CUDA_TRY(h, launch_synth_input(h->sws.y_bf.p, (long long)N * K * h->Cy, st, a.io));
                break;
            case ST_UNSHUF:
                CUDA_TRY(h, launch_synth_unshuffle(h->sws.emb, h->vecs["mask_token"], h->vecs["decoder_pos_embed"], h->sws.x, h->sws.x_bf.p,
                                                   h->sws.ln_stats, N, K, h->L, h->Dd, st, a.io));
                break;
            case ST_ATTN32:
                CUDA_TRY(h, launch_attention_hd32(h->sws.qkv.p, h->sws.attn.p, N, h->L + 1, h->syn_heads, 1.0f / sqrtf(32.0f), st));
                break;
            case ST_UNPATCH:
                CUDA_TRY(h, launch_synth_unpatchify(h->sws.pred.p, N, h->cfg.patch_size, h->grid_w, st, a.io));
                break;
            case ST_YDEC: {
                const CdfTables& t = h->cdf[TMAE_MODEL_GAUSSIAN];
                const int per_slice = h->sc * K;
                RansDecArgs d;
                d.cdf = t.cdf; d.entries = t.entries; d.n_tab = t.n;
                d.idx_stride = (long long)h->Cy * K;
                d.symbols = h->cws.ysym; d.sym_stride = (long long)h->Cy * K;
                d.n_streams = N; d.begin = sp.slice * per_slice; d.end = (sp.slice + sp.gc_slices) * per_slice;
                d.init = sp.slice == 0; d.fin = sp.slice + sp.gc_slices == h->nsl; d.status_reset = 0;
                d.state = h->cws.state;
                d.lanes = sp.lanes;
                d.io = a.io; d.io_stream = 1;
                CUDA_TRY(h, launch_rans_decode(d, st));
                break;
            }
        }
        if (h->profiling && run_end) CUDA_TRY(h, cudaEventRecord(h->prof[h->prof_used - 1].end, st));
    }
    return TMAE_OK;
}

int copy_outputs(tmae_handle* h, int N, const tmae_outputs* out, bool rate_half, bool encoder_half, cudaStream_t st) {
    if (!out) return TMAE_OK;
    Workspace& w = h->ws;
    const size_t rk = (size_t)N * h->K;
    if (encoder_half && out->ids_keep)
        CUDA_TRY(h, cudaMemcpyAsync(out->ids_keep, w.ids_keep, rk * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    if (rate_half) {
        if (out->y) CUDA_TRY(h, cudaMemcpyAsync(out->y, w.y, rk * h->Cy * 4, cudaMemcpyDeviceToDevice, st));
        if (out->z) CUDA_TRY(h, cudaMemcpyAsync(out->z, w.z, (size_t)N * h->s4 * h->s4 * h->Cz * 4, cudaMemcpyDeviceToDevice, st));
        if (out->mu) CUDA_TRY(h, cudaMemcpyAsync(out->mu, w.mu, rk * h->Cy * 4, cudaMemcpyDeviceToDevice, st));
        if (out->sigma) CUDA_TRY(h, cudaMemcpyAsync(out->sigma, w.sigma, rk * h->Cy * 4, cudaMemcpyDeviceToDevice, st));
        if (out->y_hat) CUDA_TRY(h, cudaMemcpyAsync(out->y_hat, w.yhat, rk * h->Cy * 4, cudaMemcpyDeviceToDevice, st));
    }
    return TMAE_OK;
}

// Stage `stage` of a plan.  Its first call runs plain launches (they set one-time function attributes), the second captures
// the stage into a CUDA graph and every later call replays that graph; with graphs off (TMAE_NO_GRAPH) or profiling on,
// every call runs plain launches.  The graph reads the per-call pointers `hio` from the device IoBlock `io`, uploaded on
// each call, so one capture serves every call of the plan.
// forward: the whole forward plan.  Its graph ends with the output copies (launch_copy_outputs); its plain launches read
// imgs, scores and the outputs from `hio` on the host and copy with copy_outputs.
int run_stage(tmae_handle* h, Plan& pl, int stage, const IoBlock& hio, IoBlock* io, cudaStream_t st, bool forward = false) {
    RunArgs a;
    a.begin = pl.stage_begin[stage]; a.end = pl.stage_begin[stage + 1];
    const bool replay = h->use_graph && !h->profiling && pl.stage_calls[stage]++ > 0;
    if (forward && !replay) {
        a.imgs = hio.imgs; a.scores = hio.scores; a.out = &hio.out;
        const int rc = run_steps(h, pl, a, st);
        return rc ? rc : copy_outputs(h, pl.N, &hio.out, true, true, st);
    }
    CUDA_TRY(h, cudaMemcpyAsync(io, &hio, sizeof(hio), cudaMemcpyHostToDevice, st));   // pageable source: staged before return
    a.io = io;
    if (!replay) return run_steps(h, pl, a, st);
    if (!pl.stage_graph[stage]) {
        if (!h->cap_stream) CUDA_TRY(h, cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
        CUDA_TRY(h, cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
        int rc = run_steps(h, pl, a, h->cap_stream);
        if (rc == TMAE_OK && forward) {
            const Workspace& w = h->ws;
            const int N = pl.N;
            cudaError_t e = launch_copy_outputs(io, w.y, w.z, w.mu, w.sigma, w.yhat, w.ids_keep, (long long)N * h->K * h->Cy,
                                                (long long)N * h->s4 * h->s4 * h->Cz, (long long)N * h->K, h->cap_stream);
            if (e != cudaSuccess) rc = fail(h, TMAE_ECUDA, "copy_outputs capture: %s", cudaGetErrorString(e));
        }
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamEndCapture(h->cap_stream, &g);
        if (rc != TMAE_OK) { if (g) cudaGraphDestroy(g); return rc; }
        if (e != cudaSuccess || !g) return fail(h, TMAE_ECUDA, "graph capture failed: %s", cudaGetErrorString(e));
        e = cudaGraphInstantiate(&pl.stage_graph[stage], g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) { pl.stage_graph[stage] = nullptr; return fail(h, TMAE_ECUDA, "graph instantiate failed: %s", cudaGetErrorString(e)); }
    }
    CUDA_TRY(h, cudaGraphLaunch(pl.stage_graph[stage], st));
    return TMAE_OK;
}

// The whole forward from the caller's pointers (tmae_forward, tmae_forward_host).
int run_forward(tmae_handle* h, Plan& pl, const float* imgs, const float* scores, const tmae_outputs* out, cudaStream_t st) {
    IoBlock hio;
    memset(&hio, 0, sizeof(hio));
    hio.imgs = imgs; hio.scores = scores;
    if (out) hio.out = *out;
    if (h->profiling) h->prof_used = 0;
    return run_stage(h, pl, 0, hio, h->ws.io, st, true);
}

// The per-call pointers of a decode stage: symbols in; z_hat, indexes, y_hat, mu, sigma out.
IoBlock decode_io(const int32_t* z_symbols, const int32_t* y_symbols, const tmae_outputs* out) {
    IoBlock hio;
    memset(&hio, 0, sizeof(hio));
    hio.out.z_hat = out->z_hat; hio.out.y_indexes = out->y_indexes;          // only the outputs a decode produces
    hio.out.y_hat = out->y_hat; hio.out.mu = out->mu; hio.out.sigma = out->sigma;
    hio.z_symbols = z_symbols; hio.y_symbols = y_symbols;
    return hio;
}

int check_ready(tmae_handle* h, int N) {
    if (!h) return TMAE_EINVAL;
    h->dec_next = -1;                // any other call on the handle ends a decode in progress
    if (!h->finalized) return fail(h, TMAE_ESTATE, "weights not finalized (call tmae_finalize_weights)");
    if (N <= 0) return fail(h, TMAE_EINVAL, "batch size must be positive");
    return TMAE_OK;
}

}  // namespace

// =========================================================================================================
// C ABI
// =========================================================================================================
extern "C" {

int tmae_abi_version(void) { return TMAE_ABI_VERSION; }

const char* tmae_last_error(const tmae_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int tmae_create(const tmae_config* cfg, tmae_handle** out) {
    if (!cfg || !out) return fail(nullptr, TMAE_EINVAL, "null argument");
    *out = nullptr;
    std::unique_ptr<tmae_handle> h(new tmae_handle());
    h->cfg = *cfg;
    if (h->cfg.ln_eps <= 0.f) h->cfg.ln_eps = 1e-6f;
    if (h->cfg.mlp_ratio <= 0.f) h->cfg.mlp_ratio = 4.0f;
    int rc = derive_geometry(h.get());
    if (rc) return rc;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, TMAE_ECUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    e = cudaGetDevice(&h->dev);
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, h->dev);
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, TMAE_ECUDA, "device '%s' is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
        return fail(nullptr, TMAE_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
    h->encode = reinterpret_cast<PFN_encodeTiled>(fn);
    e = gemm_tc_configure();
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "gemm configure: %s", cudaGetErrorString(e));
    e = attention_configure(h->T);
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "attention configure: %s", cudaGetErrorString(e));
    h->use_graph = getenv("TMAE_NO_GRAPH") == nullptr;
    h->precise_enc = (h->cfg.flags & TMAE_FLAG_PRECISE_ALL) != 0;
    h->precise_rate = h->precise_enc || (h->cfg.flags & TMAE_FLAG_PRECISE_RATE) != 0;
    h->planes = (h->cfg.flags & TMAE_FLAG_PRECISE_X6) ? 3 : 2;
    // the fold needs the thread-per-row TMA-store epilogue; the CUDA-core checker keeps the stand-alone LayerNorm path
    h->ln_fold = !h->precise_enc && !(h->cfg.flags & TMAE_FLAG_DEBUG_SIMT) && !getenv("TMAE_NO_LN_FOLD") && !getenv("TMAE_NO_TMA_STORE");
    h->gc_fuse = !h->precise_rate && !(h->cfg.flags & TMAE_FLAG_DEBUG_SIMT) && !getenv("TMAE_NO_GC_FUSE") && h->sc % 16 == 0;
    *out = h.release();
    return TMAE_OK;
}

void tmae_destroy(tmae_handle* h) {
    if (!h) return;
    cudaDeviceSynchronize();
    for (auto& kv : h->raw) cudaFree(kv.second.ptr);
    drop_plans(h, DEP_ALL);
    for (CdfTables& t : h->cdf) rans_free_tables(&t);
    free_pool(h->cws.allocs);
    free_pool(h->sws.allocs);
    if (h->cws.enc) cudaFree(h->cws.enc);
    if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
    if (h->scale_table) cudaFree(h->scale_table);
    free_pool(h->ws.allocs);
    free_pool(h->weight_allocs);
    for (ProfRecord& r : h->prof) { cudaEventDestroy(r.begin); cudaEventDestroy(r.end); }
    delete h;
}

int tmae_set_weight(tmae_handle* h, const char* name, const void* data, int dtype, int ndim, const int64_t* shape,
                    int* ignored) {
    if (!h || !name || !data || ndim < 0 || (ndim > 0 && !shape)) return fail(h, TMAE_EINVAL, "null/invalid argument");
    if (ignored) *ignored = 0;
    const std::string n(name);
    if (!name_is_needed(h, n)) { if (ignored) *ignored = 1; return TMAE_OK; }
    if (dtype != TMAE_F32) return fail(h, TMAE_EINVAL, "weight '%s': only f32 weights are accepted", name);
    RawTensor t;
    t.numel = 1;
    for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); t.numel *= (size_t)shape[i]; }
    void* p = nullptr;
    CUDA_TRY(h, cudaMalloc(&p, t.numel * sizeof(float) + 16));
    t.ptr = reinterpret_cast<float*>(p);
    cudaError_t e = cudaMemcpy(t.ptr, data, t.numel * sizeof(float), cudaMemcpyDefault);
    if (e != cudaSuccess) { cudaFree(p); return fail(h, TMAE_ECUDA, "copy of weight '%s' failed: %s", name, cudaGetErrorString(e)); }
    auto it = h->raw.find(n);
    if (it != h->raw.end()) cudaFree(it->second.ptr);
    h->raw[n] = t;
    h->finalized = false;
    return TMAE_OK;
}

int tmae_finalize_weights(tmae_handle* h) {
    if (!h) return TMAE_EINVAL;
    // re-finalize: drop previous packs
    drop_plans(h, DEP_ALL);
    h->dec_next = -1;
    free_pool(h->weight_allocs);
    h->layers.clear();
    h->vecs.clear();
    h->eb_tab = nullptr;
    const int C = h->C, one[1] = {0};
    (void)one;
    int rc;
    if ((rc = keep_vec(h, "cls_token", C))) return rc;
    if ((rc = keep_vec(h, "encoder_pos_embed", (size_t)(h->L + 1) * C))) return rc;
    { int sg[1] = {h->patch_dim}; if ((rc = pack_layer(h, "encoder_embed.proj", "encoder_embed.proj", C, h->patch_dim, 1, 1, sg, 0, h->precise_enc))) return rc; }
    for (int i = 0; i < h->cfg.encoder_depth; ++i) {
        const std::string pre = "encoder_blocks." + std::to_string(i);
        for (const char* nm : {".norm1.weight", ".norm1.bias", ".norm2.weight", ".norm2.bias"})
            if ((rc = keep_vec(h, pre + nm, C))) return rc;
        int sgC[1] = {C}, sgM[1] = {h->mlp};
        if ((rc = pack_layer(h, pre + ".attn.qkv", pre + ".attn.qkv", 3 * C, C, 1, 1, sgC, 0, h->precise_enc,
                             (h->ln_fold && i > 0) ? pre + ".norm1" : std::string()))) return rc;
        if ((rc = pack_layer(h, pre + ".attn.proj", pre + ".attn.proj", C, C, 1, 1, sgC, 0, h->precise_enc))) return rc;
        if ((rc = pack_layer(h, pre + ".mlp.fc1", pre + ".mlp.fc1", h->mlp, C, 1, 1, sgC, 0, h->precise_enc,
                             h->ln_fold ? pre + ".norm2" : std::string()))) return rc;
        if ((rc = pack_layer(h, pre + ".mlp.fc2", pre + ".mlp.fc2", C, h->mlp, 1, 1, sgM, 0, h->precise_enc))) return rc;
    }
    if ((rc = keep_vec(h, "encoder_norm.weight", C))) return rc;
    if ((rc = keep_vec(h, "encoder_norm.bias", C))) return rc;
    for (int l = 0; l < 4; ++l) {
        int sg[1] = {h->ga_ch[l]};
        const std::string nm = "g_a." + std::to_string(2 * l);
        if ((rc = pack_layer(h, nm, nm, h->ga_ch[l + 1], h->ga_ch[l], 1, 1, sg, 0, h->precise_rate))) return rc;
    }
    {
        int ci[5], co[5], aux[5];
        ha_layers(h, ci, co, aux);
        for (int l = 0; l < 5; ++l) {
            int sg[1] = {ci[l]};
            const std::string nm = "h_a." + std::to_string(2 * l);
            if ((rc = pack_layer(h, nm, nm, co[l], ci[l], 9, 1, sg, 0, h->precise_rate))) return rc;
        }
        hs_layers(h, ci, co, aux);
        for (const char* net : {"h_s_mean", "h_s_scale"})
            for (int l = 0; l < 5; ++l) {
                int sg[1] = {ci[l]};
                const std::string key = std::string(net) + "." + std::to_string(2 * l);
                const std::string wname = aux[l] == 2 ? key + ".0" : key;      // subpel = Sequential(conv, PixelShuffle)
                if ((rc = pack_layer(h, key, wname, co[l] * aux[l] * aux[l], ci[l], 9, 1, sg, aux[l] == 2, h->precise_rate))) return rc;
            }
    }
    for (int i = 0; i < h->nsl; ++i) {
        const int sup = i < h->nsl / 2 ? i : h->nsl / 2;
        int ch[6];
        cc_channels(h, ch, i, false);
        for (const char* net : {"cc_transform_mean.", "cc_transform_scale."})
            for (int l = 0; l < 5; ++l) {
                const std::string nm = std::string(net) + std::to_string(i) + "." + std::to_string(2 * l);
                int sg[3] = {ch[l], 0, 0};
                int nseg = 1;
                if (l == 0 && sup > 0) { sg[0] = h->Cy; sg[1] = h->sc * sup; nseg = 2; }
                if ((rc = pack_layer(h, nm, nm, ch[l + 1], ch[l], 9, nseg, sg, 0, h->precise_rate))) return rc;
            }
        if (h->gc_fuse) {      // cc_transform_mean[i].8 and cc_transform_scale[i].8 as one block-diagonal layer "gc.<i>"
            const RawTensor *wa = nullptr, *wb = nullptr, *ba = nullptr, *bb = nullptr;
            const std::string ma = "cc_transform_mean." + std::to_string(i) + ".8", mb = "cc_transform_scale." + std::to_string(i) + ".8";
            if ((rc = need_raw(h, ma + ".weight", (size_t)h->sc * ch[4] * 9, &wa)) || (rc = need_raw(h, mb + ".weight", (size_t)h->sc * ch[4] * 9, &wb)) ||
                (rc = need_raw(h, ma + ".bias", (size_t)h->sc, &ba)) || (rc = need_raw(h, mb + ".bias", (size_t)h->sc, &bb))) return rc;
            RawTensor wt, bt;
            wt.numel = (size_t)2 * h->sc * 2 * ch[4] * 9; wt.shape = {2 * h->sc, 2 * ch[4], 3, 3};
            bt.numel = (size_t)2 * h->sc; bt.shape = {2 * h->sc};
            CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&wt.ptr), wt.numel * sizeof(float)));
            CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&bt.ptr), bt.numel * sizeof(float)));
            CUDA_TRY(h, launch_build_blockdiag2(wa->ptr, wb->ptr, ba->ptr, bb->ptr, wt.ptr, bt.ptr, h->sc, ch[4], 9, 0));
            const std::string key = "gc." + std::to_string(i);
            h->raw[key + ".weight"] = wt;          // freed with the other raw tensors at the end of finalize
            h->raw[key + ".bias"] = bt;
            int sg[3] = {ch[4], ch[4], 0};
            if ((rc = pack_layer(h, key, key, 2 * h->sc, 2 * ch[4], 9, 2, sg, 0, false))) return rc;
        }
        int lch[6];
        cc_channels(h, lch, i, true);
        for (int l = 0; l < 5; ++l) {
            const std::string nm = "lrp_transform." + std::to_string(i) + "." + std::to_string(2 * l);
            int sg[3] = {lch[l], 0, 0};
            int nseg = 1;
            if (l == 0) {
                sg[0] = h->Cy;
                if (i < h->nsl / 2) { sg[1] = h->sc * (i + 1); nseg = 2; }
                else { sg[1] = h->sc * sup; sg[2] = h->sc; nseg = 3; }
            }
            if ((rc = pack_layer(h, nm, nm, lch[l + 1], lch[l], 9, nseg, sg, 0, h->precise_rate))) return rc;
        }
    }
    {   // factorized prior table
        const int Cz = h->Cz;
        const size_t sizes[15] = {3, 3, 3, 9, 3, 3, 9, 3, 3, 9, 3, 3, 3, 1, 3};
        const char* names[15] = {"_matrix0", "_bias0", "_factor0", "_matrix1", "_bias1", "_factor1", "_matrix2", "_bias2",
                                 "_factor2", "_matrix3", "_bias3", "_factor3", "_matrix4", "_bias4", "quantiles"};
        const float* ptrs[15];
        for (int i = 0; i < 15; ++i) {
            const RawTensor* r = nullptr;
            if ((rc = need_raw(h, std::string("entropy_bottleneck.") + names[i], sizes[i] * Cz, &r))) return rc;
            ptrs[i] = r->ptr;
        }
        if ((rc = dev_alloc(h, h->weight_allocs, &h->eb_tab, (size_t)Cz * 64))) return rc;
        CUDA_TRY(h, launch_eb_table(ptrs, h->eb_tab, Cz, 0));
    }
    if (h->syn_depth > 0 && (rc = pack_synthesis(h))) return rc;
    CUDA_TRY(h, cudaDeviceSynchronize());
    for (auto& kv : h->raw) cudaFree(kv.second.ptr);
    h->raw.clear();
    h->finalized = true;
    return TMAE_OK;
}

size_t tmae_workspace_bytes(const tmae_handle* h, int N) { return h && N > 0 ? workspace_bytes_estimate(h, N) : 0; }

int tmae_reserve(tmae_handle* h, int N) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    Plan* pl = nullptr;
    return get_plan(h, PLAN_FORWARD, N, &pl);
}

int tmae_attention_plan(int T, int H, int N, int mode, int* out) {
    if (!out || T <= 0 || H <= 0 || N <= 0 || mode < 1 || mode > 3) return fail(nullptr, TMAE_EINVAL, "tmae_attention_plan: invalid argument");
    attention_tc_describe(T, H, N, mode, out);
    return TMAE_OK;
}

int tmae_conv_geometry(int s, int n_img, int* out) {
    ConvGeom cg;
    if (!out || !conv_geom(s, n_img, &cg)) return TMAE_EINVAL;
    out[0] = cg.box_y; out[1] = cg.box_n; out[2] = cg.y_tiles; out[3] = cg.m_tiles; out[4] = cg.rows_used; out[5] = cg.reuse_ok ? 1 : 0;
    return TMAE_OK;
}

int tmae_launch_count(tmae_handle* h, int N) {
    Plan* pl = nullptr;
    if (check_ready(h, N) || get_plan(h, PLAN_FORWARD, N, &pl)) return -1;
    return (int)pl->steps.size();
}

int tmae_forward(tmae_handle* h, const float* imgs, const float* scores, int N, const tmae_outputs* out, void* stream) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!imgs || !scores) return fail(h, TMAE_EINVAL, "imgs / scores must not be null");
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_FORWARD, N, &pl))) return rc;
    return run_forward(h, *pl, imgs, scores, out, reinterpret_cast<cudaStream_t>(stream));
}

int tmae_forward_encoder(tmae_handle* h, const float* imgs, const float* scores, int N, const tmae_outputs* out,
                         void* stream) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!imgs || !scores) return fail(h, TMAE_EINVAL, "imgs / scores must not be null");
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_FORWARD, N, &pl))) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    RunArgs a;
    a.imgs = imgs; a.scores = scores; a.out = out; a.begin = 0; a.end = pl->encoder_end_step;
    if (h->profiling) h->prof_used = 0;
    if ((rc = run_steps(h, *pl, a, st))) return rc;
    return copy_outputs(h, N, out, false, true, st);
}

int tmae_forward_from_latent(tmae_handle* h, const float* y, int N, const tmae_outputs* out, void* stream) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!y) return fail(h, TMAE_EINVAL, "y must not be null");
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_FORWARD, N, &pl))) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Workspace& w = h->ws;
    const size_t rk = (size_t)N * h->K;
    CUDA_TRY(h, cudaMemsetAsync(w.rate_acc, 0, sizeof(double) * N, st));
    CUDA_TRY(h, cudaMemcpyAsync(w.y, y, rk * h->Cy * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(h, launch_f32_to_bf16(w.y, w.y_bf.p, (long long)rk * h->Cy, w.y_bf.lo, st));
    RunArgs a;
    a.out = out; a.begin = pl->first_rate_step; a.end = (int)pl->steps.size();
    if (h->profiling) h->prof_used = 0;
    if ((rc = run_steps(h, *pl, a, st))) return rc;
    return copy_outputs(h, N, out, true, false, st);
}

int tmae_forward_from_latent_forced(tmae_handle* h, const float* y, const float* y_hat_support, int N, const tmae_outputs* out,
                                    void* stream) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!y || !y_hat_support) return fail(h, TMAE_EINVAL, "y / y_hat_support must not be null");
    if (h->cfg.flags & TMAE_FLAG_SKIP_DEAD_LRP) return fail(h, TMAE_EINVAL, "forced support needs every lrp_transform");
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_FORCED, N, &pl))) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Workspace& w = h->ws;
    const size_t rk = (size_t)N * h->K;
    CUDA_TRY(h, cudaMemsetAsync(w.rate_acc, 0, sizeof(double) * N, st));
    CUDA_TRY(h, cudaMemcpyAsync(w.y, y, rk * h->Cy * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(h, cudaMemcpyAsync(w.yhat_force, y_hat_support, rk * h->Cy * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(h, launch_f32_to_bf16(w.y, w.y_bf.p, (long long)rk * h->Cy, w.y_bf.lo, st));
    RunArgs a;
    a.out = out; a.begin = pl->first_rate_step; a.end = (int)pl->steps.size();
    const bool prof = h->profiling;
    h->profiling = false;
    rc = run_steps(h, *pl, a, st);
    h->profiling = prof;
    if (rc) return rc;
    return copy_outputs(h, N, out, true, false, st);
}

int tmae_forward_host(tmae_handle* h, const float* h_imgs, const float* h_scores, int N, const tmae_host_outputs* hout,
                      const tmae_outputs* out, void* stream) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!h_imgs || !h_scores) return fail(h, TMAE_EINVAL, "h_imgs / h_scores must not be null");
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_FORWARD, N, &pl))) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Workspace& w = h->ws;
    const size_t img_elems = (size_t)N * h->cfg.in_chans * h->cfg.img_size * h->cfg.img_size;
    CUDA_TRY(h, cudaMemcpyAsync(w.st_imgs, h_imgs, img_elems * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaMemcpyAsync(w.st_scores, h_scores, (size_t)N * h->L * sizeof(float), cudaMemcpyHostToDevice, st));
    tmae_outputs o = out ? *out : tmae_outputs{};
    static const tmae_host_outputs kNoHost = {};
    const tmae_host_outputs& ho = hout ? *hout : kNoHost;
    if (!o.bpp) o.bpp = w.bpp;
    if (!o.rate_sums) o.rate_sums = w.rate_sums;
    // results the host asked for are produced into device staging buffers (unless the caller also gave device buffers)
    if (ho.y_likelihoods && !o.y_likelihoods) o.y_likelihoods = w.st_ylik;
    if (ho.z_likelihoods && !o.z_likelihoods) o.z_likelihoods = w.st_zlik;
    if (ho.y_symbols && !o.y_symbols_i16) o.y_symbols_i16 = w.st_ysym;
    if (ho.z_symbols && !o.z_symbols_i16) o.z_symbols_i16 = w.st_zsym;
    if (ho.ids_restore && !o.ids_restore) o.ids_restore = w.st_ids_restore;
    if ((rc = run_forward(h, *pl, w.st_imgs, w.st_scores, &o, st))) return rc;
    const size_t ny = (size_t)N * h->K * h->Cy, nz = (size_t)N * h->s4 * h->s4 * h->Cz;
    if (ho.bpp) CUDA_TRY(h, cudaMemcpyAsync(ho.bpp, o.bpp, (size_t)N * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (ho.rate_sums) CUDA_TRY(h, cudaMemcpyAsync(ho.rate_sums, o.rate_sums, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (ho.y_likelihoods) CUDA_TRY(h, cudaMemcpyAsync(ho.y_likelihoods, o.y_likelihoods, ny * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (ho.z_likelihoods) CUDA_TRY(h, cudaMemcpyAsync(ho.z_likelihoods, o.z_likelihoods, nz * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (ho.y_symbols) CUDA_TRY(h, cudaMemcpyAsync(ho.y_symbols, o.y_symbols_i16, ny * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
    if (ho.z_symbols) CUDA_TRY(h, cudaMemcpyAsync(ho.z_symbols, o.z_symbols_i16, nz * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
    if (ho.ids_restore) CUDA_TRY(h, cudaMemcpyAsync(ho.ids_restore, o.ids_restore, (size_t)N * h->L * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    return TMAE_OK;
}

int tmae_set_scale_table(tmae_handle* h, const float* table, int n) {
    if (!h || !table || n < 2 || n > 256) return fail(h, TMAE_EINVAL, "scale table: need 2..256 ascending entries");
    if (!h->scale_table) CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&h->scale_table), 256 * sizeof(float)));
    CUDA_TRY(h, cudaDeviceSynchronize());
    CUDA_TRY(h, cudaMemcpy(h->scale_table, table, (size_t)n * sizeof(float), cudaMemcpyDefault));
    h->n_scale_table = n;
    drop_plans(h, DEP_SCALE);        // plans and their graphs carry the table pointer / length
    h->dec_next = -1;
    return TMAE_OK;
}

// ---- decode (MCM.decompress without the range coder) ---------------------------------------------------
int tmae_decode_groups(int num_slices, int* first_slice, int* n_slices, int capacity) {
    if (num_slices <= 0 || num_slices % 2 != 0) return -TMAE_EINVAL;
    std::vector<std::pair<int, int>> g;
    slice_groups(num_slices, g);
    if ((first_slice || n_slices) && capacity < (int)g.size()) return -TMAE_EINVAL;
    for (size_t i = 0; i < g.size(); ++i) {
        if (first_slice) first_slice[i] = g[i].first;
        if (n_slices) n_slices[i] = g[i].second;
    }
    return (int)g.size();
}

int tmae_decode_begin(tmae_handle* h, const int32_t* z_symbols, int N, const tmae_outputs* out, void* stream) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!z_symbols || !out || !out->y_indexes) return fail(h, TMAE_EINVAL, "z_symbols, out and out->y_indexes must not be null");
    if (!h->scale_table) return fail(h, TMAE_ESTATE, "decoding needs the scale table (call tmae_set_scale_table first)");
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_DECODE, N, &pl))) return rc;
    if (h->profiling) h->prof_used = 0;
    if ((rc = run_stage(h, *pl, 0, decode_io(z_symbols, nullptr, out), h->ws.io, reinterpret_cast<cudaStream_t>(stream)))) return rc;
    h->dec_N = N;
    h->dec_next = 0;
    return TMAE_OK;
}

int tmae_decode_step(tmae_handle* h, int group, const int32_t* y_symbols, const tmae_outputs* out, void* stream) {
    if (!h) return TMAE_EINVAL;
    if (!y_symbols || !out || !out->y_indexes) return fail(h, TMAE_EINVAL, "y_symbols, out and out->y_indexes must not be null");
    const int expected = h->dec_next;
    auto it = h->plans.find(PlanKey(PLAN_DECODE, h->dec_N, 0, 0));
    h->dec_next = -1;                // an out-of-order step ends the decode as well
    if (expected < 0 || group != expected || it == h->plans.end())
        return fail(h, TMAE_ESTATE, "decode step %d out of order (expected %s%d): steps follow tmae_decode_begin in group order, "
                    "and any other call on the handle in between ends the decode", group, expected < 0 ? "a new tmae_decode_begin, not step " : "step ",
                    expected < 0 ? group : expected);
    Plan& pl = *it->second;
    const int rc = run_stage(h, pl, group + 1, decode_io(nullptr, y_symbols, out), h->ws.io, reinterpret_cast<cudaStream_t>(stream));
    if (rc) return rc;
    if (group + 2 < (int)pl.stage_begin.size() - 1) h->dec_next = group + 1;
    return TMAE_OK;
}

// ---- synthesis (recon.synthesize on the engine) ---------------------------------------------------------
int tmae_enable_synthesis(tmae_handle* h, int decoder_depth, int decoder_num_heads) {
    if (!h) return TMAE_EINVAL;
    const int Dd = h->cfg.decoder_embed_dim;
    if (decoder_depth < 1) return fail(h, TMAE_EINVAL, "decoder_depth must be >= 1 (got %d)", decoder_depth);
    if (decoder_num_heads < 1 || Dd % decoder_num_heads != 0)
        return fail(h, TMAE_EINVAL, "decoder_num_heads %d does not divide decoder_embed_dim %d", decoder_num_heads, Dd);
    if (Dd / decoder_num_heads != 32)
        return fail(h, TMAE_EINVAL, "synthesis supports a decoder head dim of 32 only (decoder_embed_dim %d / %d heads = %d)", Dd,
                    decoder_num_heads, Dd / decoder_num_heads);
    if ((h->cfg.flags & TMAE_FLAG_DEBUG_SIMT) || getenv("TMAE_NO_TMA_STORE"))
        return fail(h, TMAE_EINVAL, "synthesis folds its LayerNorms into the TMA-store phase of the tensor-core GEMMs: not available with "
                    "TMAE_FLAG_DEBUG_SIMT or TMAE_NO_TMA_STORE");
    const int mlp = (int)(Dd * h->cfg.mlp_ratio);
    if (mlp <= 0 || mlp % 32 != 0) return fail(h, TMAE_EINVAL, "decoder MLP width %d must be a positive multiple of 32", mlp);
    if (!attention_hd32_supported(h->L + 1))
        return fail(h, TMAE_EINVAL, "synthesis attention over %d tokens does not fit shared memory", h->L + 1);
    h->dec_next = -1;
    drop_plans(h, DEP_SYNTH);
    if (decoder_depth != h->syn_depth || Dd != h->Dd || mlp != h->syn_mlp) {   // buffers sized for another decoder
        free_pool(h->sws.allocs);
        h->sws = SynthWorkspace();
    }
    h->syn_depth = decoder_depth;
    h->syn_heads = decoder_num_heads;
    h->Dd = Dd;
    h->syn_mlp = mlp;
    h->syn_out = h->cfg.patch_size * h->cfg.patch_size * h->cfg.in_chans;
    h->finalized = false;            // the decoder-side tensors must be packed
    return TMAE_OK;
}

int tmae_synthesize(tmae_handle* h, const float* y_hat, const int64_t* ids_restore, int N, float* x_hat, void* stream) {
    if (!h) return TMAE_EINVAL;
    if (h->syn_depth == 0) { h->dec_next = -1; return fail(h, TMAE_ESTATE, "synthesis is not enabled (call tmae_enable_synthesis)"); }
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!y_hat || !ids_restore || !x_hat) return fail(h, TMAE_EINVAL, "y_hat, ids_restore and x_hat must not be null");
    if (((reinterpret_cast<uintptr_t>(y_hat) | reinterpret_cast<uintptr_t>(x_hat)) & 15) != 0)
        return fail(h, TMAE_EINVAL, "y_hat and x_hat must be 16-byte aligned");
    if (h->cfg.in_chans != 3) return fail(h, TMAE_EINVAL, "synthesis writes 3-channel images (in_chans %d)", h->cfg.in_chans);
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_SYNTH, N, &pl))) return rc;
    IoBlock hio;
    memset(&hio, 0, sizeof(hio));
    hio.syn_y_hat = y_hat; hio.syn_ids = ids_restore; hio.syn_x_hat = x_hat;
    if (h->profiling) h->prof_used = 0;
    return run_stage(h, *pl, 0, hio, h->sws.io, reinterpret_cast<cudaStream_t>(stream));
}

// ---- entropy coder (compressai's rANS format) -----------------------------------------------------------
int tmae_pmf_to_quantized_cdf(const float* h_pmf, int n, int32_t* h_cdf) {
    if (!h_pmf || !h_cdf || n < 1) return fail(nullptr, TMAE_EINVAL, "pmf_to_quantized_cdf: null pointer or n < 1");
    const int rc = pmf_to_quantized_cdf(h_pmf, n, h_cdf);
    if (rc) return fail(nullptr, rc, "pmf_to_quantized_cdf: the pmf must be finite, non-negative, not all zero, with at most 65536 bins");
    return TMAE_OK;
}

int64_t tmae_rans_bound(int64_t n_symbols) { return n_symbols < 0 || n_symbols > ((int64_t)1 << 40) ? -1 : rans_bound_bytes(n_symbols); }

int tmae_set_cdf_tables(tmae_handle* h, int model, const int32_t* cdf, int n_tables, int stride, const int32_t* cdf_lengths,
                        const int32_t* offsets) {
    if (!h) return TMAE_EINVAL;
    h->dec_next = -1;
    if (model != TMAE_MODEL_GAUSSIAN && model != TMAE_MODEL_BOTTLENECK) return fail(h, TMAE_EINVAL, "unknown entropy model %d", model);
    if (!cdf || !cdf_lengths || !offsets || n_tables < 1 || stride < 3)
        return fail(h, TMAE_EINVAL, "cdf tables: null pointer, n_tables < 1 or stride < 3");
    if ((size_t)n_tables * stride > ((size_t)1 << 30)) return fail(h, TMAE_EINVAL, "cdf tables too large");
    if (model == TMAE_MODEL_BOTTLENECK && n_tables != h->Cz)
        return fail(h, TMAE_EINVAL, "bottleneck tables: %d given, one per channel (%d) needed", n_tables, h->Cz);
    std::vector<int32_t> c((size_t)n_tables * stride), len(n_tables), off(n_tables);
    CUDA_TRY(h, cudaDeviceSynchronize());           // host or device pointers, possibly written by pending work
    CUDA_TRY(h, cudaMemcpy(c.data(), cdf, c.size() * 4, cudaMemcpyDefault));
    CUDA_TRY(h, cudaMemcpy(len.data(), cdf_lengths, len.size() * 4, cudaMemcpyDefault));
    CUDA_TRY(h, cudaMemcpy(off.data(), offsets, off.size() * 4, cudaMemcpyDefault));
    CdfTables t;
    char err[256] = {0};
    const int rc = rans_build_tables(c.data(), n_tables, stride, len.data(), off.data(), &t, err, sizeof(err));
    if (rc) return fail(h, rc, "cdf tables: %s", err);
    drop_plans(h, DEP_CDF);                          // their graphs captured the previous tables
    rans_free_tables(&h->cdf[model]);
    h->cdf[model] = t;
    return TMAE_OK;
}

namespace {
int coder_tables(tmae_handle* h, int model, const CdfTables** out) {
    if (!h) return TMAE_EINVAL;
    h->dec_next = -1;                // any other call on the handle ends a decode in progress
    if (model != TMAE_MODEL_GAUSSIAN && model != TMAE_MODEL_BOTTLENECK) return fail(h, TMAE_EINVAL, "unknown entropy model %d", model);
    if (!h->cdf[model].n) return fail(h, TMAE_ESTATE, "no cdf tables for model %d (call tmae_set_cdf_tables first)", model);
    *out = &h->cdf[model];
    return TMAE_OK;
}
}  // namespace

namespace {
bool bad_lanes(int lanes) { return lanes < 1 || lanes > 32; }

// lanes = 0: compressai's format, else the laned format
int rans_encode_impl(tmae_handle* h, int model, const int32_t* symbols, const int32_t* indexes, int n_streams, int n_per_stream,
                     int lanes, uint8_t* out, int64_t capacity, int64_t* offsets, int32_t* status, void* stream) {
    const CdfTables* t = nullptr;
    int rc = coder_tables(h, model, &t);
    if (rc) return rc;
    if (n_streams < 1 || n_per_stream < 0 || (n_per_stream > 0 && (!symbols || !indexes)) || !out || !offsets || !status || capacity < 0)
        return fail(h, TMAE_EINVAL, "rans_encode: null pointer or bad size");
    if (reinterpret_cast<uintptr_t>(out) & 3) return fail(h, TMAE_EINVAL, "rans_encode: out must be 4-byte aligned");
    const int chains = lanes ? lanes : 1;           // scratch: one region per (stream, lane), sized for the longest lane
    const long long cap_words = rans_bound_bytes((n_per_stream + chains - 1) / chains) / 4;
    const size_t rec_bytes = ((size_t)n_streams * n_per_stream * sizeof(uint2) + 255) / 256 * 256;
    const size_t words_bytes = ((size_t)n_streams * chains * cap_words * 4 + 255) / 256 * 256;
    const size_t need = rec_bytes + words_bytes + (size_t)n_streams * chains * 8;
    CoderWorkspace& c = h->cws;
    if (need > c.enc_bytes) {
        if (c.enc) { cudaFree(c.enc); c.enc = nullptr; c.enc_bytes = 0; }
        cudaError_t e = cudaMalloc(&c.enc, need);
        if (e != cudaSuccess) return fail(h, TMAE_ENOMEM, "rans_encode scratch (%zu bytes): %s", need, cudaGetErrorString(e));
        c.enc_bytes = need;
    }
    char* base = static_cast<char*>(c.enc);
    CUDA_TRY(h, launch_rans_encode(symbols, indexes, n_streams, n_per_stream, lanes, *t, reinterpret_cast<uint2*>(base),
                                   reinterpret_cast<uint32_t*>(base + rec_bytes), cap_words,
                                   reinterpret_cast<long long*>(base + rec_bytes + words_bytes), out, capacity, offsets, status,
                                   reinterpret_cast<cudaStream_t>(stream)));
    return TMAE_OK;
}

int rans_decode_impl(tmae_handle* h, int model, const uint8_t* data, const int64_t* offsets, int n_streams, const int32_t* indexes,
                     int n_per_stream, int lanes, int32_t* symbols, int32_t* status, void* stream) {
    const CdfTables* t = nullptr;
    int rc = coder_tables(h, model, &t);
    if (rc) return rc;
    if (n_streams < 1 || n_per_stream < 0 || !data || !offsets || !status || (n_per_stream > 0 && (!indexes || !symbols)))
        return fail(h, TMAE_EINVAL, "rans_decode: null pointer or bad size");
    if (reinterpret_cast<uintptr_t>(data) & 3) return fail(h, TMAE_EINVAL, "rans_decode: data must be 4-byte aligned");
    RansDecArgs d;
    d.cdf = t->cdf; d.entries = t->entries; d.n_tab = t->n;
    d.lanes = lanes;
    d.data = data; d.offsets = offsets;
    d.indexes = indexes; d.idx_stride = n_per_stream;
    d.symbols = symbols; d.sym_stride = n_per_stream;
    d.n_streams = n_streams; d.begin = 0; d.end = n_per_stream;
    d.status = status;
    CUDA_TRY(h, launch_rans_decode(d, reinterpret_cast<cudaStream_t>(stream)));
    return TMAE_OK;
}

int decompress_streams_impl(tmae_handle* h, const uint8_t* y_data, const int64_t* y_offsets, int y_lanes, const uint8_t* z_data,
                            const int64_t* z_offsets, int z_lanes, int N, const tmae_outputs* out, int32_t* status, void* stream) {
    int rc = check_ready(h, N);
    if (rc) return rc;
    if (!y_data || !y_offsets || !z_data || !z_offsets || !out || !status)
        return fail(h, TMAE_EINVAL, "decompress_streams: stream pointers, out and status must not be null");
    if ((reinterpret_cast<uintptr_t>(y_data) | reinterpret_cast<uintptr_t>(z_data)) & 3)
        return fail(h, TMAE_EINVAL, "decompress_streams: stream data must be 4-byte aligned");
    if (!h->scale_table) return fail(h, TMAE_ESTATE, "decoding needs the scale table (call tmae_set_scale_table first)");
    if (!h->cdf[TMAE_MODEL_GAUSSIAN].n || !h->cdf[TMAE_MODEL_BOTTLENECK].n)
        return fail(h, TMAE_ESTATE, "decoding streams needs both cdf table sets (tmae_set_cdf_tables)");
    if (h->cdf[TMAE_MODEL_GAUSSIAN].n != h->n_scale_table)
        return fail(h, TMAE_ESTATE, "%d Gaussian cdf tables for a scale table of %d entries", h->cdf[TMAE_MODEL_GAUSSIAN].n, h->n_scale_table);
    Plan* pl = nullptr;
    if ((rc = get_plan(h, PLAN_STREAMS, N, &pl, y_lanes, z_lanes))) return rc;
    IoBlock hio = decode_io(h->cws.zsym, h->cws.ysym, out);
    if (!hio.out.y_indexes) hio.out.y_indexes = h->cws.idx;
    hio.y_data = y_data; hio.y_offsets = y_offsets; hio.z_data = z_data; hio.z_offsets = z_offsets; hio.status = status;
    if (h->profiling) h->prof_used = 0;
    return run_stage(h, *pl, 0, hio, h->ws.io, reinterpret_cast<cudaStream_t>(stream));
}
}  // namespace

int tmae_rans_encode(tmae_handle* h, int model, const int32_t* symbols, const int32_t* indexes, int n_streams, int n_per_stream,
                     uint8_t* out, int64_t capacity, int64_t* offsets, int32_t* status, void* stream) {
    return rans_encode_impl(h, model, symbols, indexes, n_streams, n_per_stream, 0, out, capacity, offsets, status, stream);
}

int tmae_rans_decode(tmae_handle* h, int model, const uint8_t* data, const int64_t* offsets, int n_streams, const int32_t* indexes,
                     int n_per_stream, int32_t* symbols, int32_t* status, void* stream) {
    return rans_decode_impl(h, model, data, offsets, n_streams, indexes, n_per_stream, 0, symbols, status, stream);
}

int tmae_decompress_streams(tmae_handle* h, const uint8_t* y_data, const int64_t* y_offsets, const uint8_t* z_data,
                            const int64_t* z_offsets, int N, const tmae_outputs* out, int32_t* status, void* stream) {
    return decompress_streams_impl(h, y_data, y_offsets, 0, z_data, z_offsets, 0, N, out, status, stream);
}

int64_t tmae_rans_bound_lanes(int64_t n_symbols, int lanes) {
    return n_symbols > ((int64_t)1 << 40) ? -1 : rans_bound_lanes_bytes(n_symbols, lanes);
}

int tmae_rans_encode_lanes(tmae_handle* h, int model, const int32_t* symbols, const int32_t* indexes, int n_streams, int n_per_stream,
                           int lanes, uint8_t* out, int64_t capacity, int64_t* offsets, int32_t* status, void* stream) {
    if (!h || bad_lanes(lanes) || !out || !offsets || !status || (n_per_stream > 0 && (!symbols || !indexes)))
        return fail(h, TMAE_EINVAL, "rans_encode_lanes: null pointer, or lanes %d outside 1..32", lanes);
    return rans_encode_impl(h, model, symbols, indexes, n_streams, n_per_stream, lanes, out, capacity, offsets, status, stream);
}

int tmae_rans_decode_lanes(tmae_handle* h, int model, const uint8_t* data, const int64_t* offsets, int n_streams,
                           const int32_t* indexes, int n_per_stream, int lanes, int32_t* symbols, int32_t* status, void* stream) {
    if (!h || bad_lanes(lanes) || !data || !offsets || !status || (n_per_stream > 0 && (!indexes || !symbols)))
        return fail(h, TMAE_EINVAL, "rans_decode_lanes: null pointer, or lanes %d outside 1..32", lanes);
    return rans_decode_impl(h, model, data, offsets, n_streams, indexes, n_per_stream, lanes, symbols, status, stream);
}

int tmae_decompress_streams_lanes(tmae_handle* h, const uint8_t* y_data, const int64_t* y_offsets, int y_lanes, const uint8_t* z_data,
                                  const int64_t* z_offsets, int z_lanes, int N, const tmae_outputs* out, int32_t* status, void* stream) {
    if (!h || bad_lanes(y_lanes) || bad_lanes(z_lanes) || !y_data || !y_offsets || !z_data || !z_offsets || !out || !status)
        return fail(h, TMAE_EINVAL, "decompress_streams_lanes: null pointer, or lanes (%d, %d) outside 1..32", y_lanes, z_lanes);
    return decompress_streams_impl(h, y_data, y_offsets, y_lanes, z_data, z_offsets, z_lanes, N, out, status, stream);
}

int tmae_pack_nchw_i32(const int32_t* nhwc, int32_t* nchw, int N, int hw, int C, void* stream) {
    if (!nhwc || !nchw || N < 0 || hw <= 0 || C <= 0) return fail(nullptr, TMAE_EINVAL, "invalid argument");
    cudaError_t e = launch_pack_nchw_i32(nhwc, nchw, N, hw, C, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "pack_nchw: %s", cudaGetErrorString(e));
    return TMAE_OK;
}

// ---- stand-alone operators -----------------------------------------------------------------------------
int tmae_mask_select(const float* scores, int N, int L, int K, int softmax_isa, int64_t* ids_shuffle,
                     int64_t* ids_restore, int64_t* ids_keep, void* stream) {
    if (!scores || N < 0 || L <= 0) return fail(nullptr, TMAE_EINVAL, "invalid argument");
    if (K > L) return fail(nullptr, TMAE_EINVAL, "Number of patches should not be greater than the length of scores");
    cudaError_t e = launch_mask_select(scores, N, L, K, softmax_isa, ids_shuffle, ids_restore, ids_keep,
                                       reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "mask_select: %s", cudaGetErrorString(e));
    return TMAE_OK;
}

int tmae_gaussian_rate(const float* y, const float* mu, const float* sigma, int64_t n, float* likelihood,
                       int32_t* symbols, float* y_hat, void* stream) {
    if (!y || !mu || !sigma || n < 0) return fail(nullptr, TMAE_EINVAL, "invalid argument");
    cudaError_t e = launch_gaussian_flat(y, mu, sigma, n, likelihood, symbols, y_hat, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "gaussian_rate: %s", cudaGetErrorString(e));
    return TMAE_OK;
}

int tmae_bottleneck_rate(tmae_handle* h, const float* z, int64_t rows, float* likelihood, int32_t* symbols, float* z_hat,
                         void* stream) {
    if (!h || !h->finalized) return fail(h, TMAE_ESTATE, "weights not finalized");
    if (!z || rows < 0) return fail(h, TMAE_EINVAL, "invalid argument");
    CUDA_TRY(h, launch_bottleneck(z, h->eb_tab, rows, h->Cz, likelihood, symbols, z_hat, nullptr, 0, 1, nullptr, 1, nullptr,
                                  reinterpret_cast<cudaStream_t>(stream)));
    return TMAE_OK;
}

// ---- patch-score generation (generate_scores_file.py:19-31) ---------------------------------------------
size_t tmae_scores_workspace_bytes(int n, int height, int width, int out_side) {
    ScoreGeom g;
    if (n < 0 || !score_geometry(height, width, out_side, &g)) return 0;
    return score_workspace_bytes(g, n);
}
int tmae_generate_scores(const uint8_t* gray, int n, int height, int width, int out_side, const tmae_score_outputs* out,
                         void* workspace, size_t workspace_bytes, void* stream) {
    ScoreGeom g;
    if (n < 0 || !out || (n > 0 && (!gray || !workspace))) return fail(nullptr, TMAE_EINVAL, "invalid argument");
    if (!score_geometry(height, width, out_side, &g))
        return fail(nullptr, TMAE_EINVAL, "score generation needs height, width >= 8 and out_side a positive multiple of 16 (got %d x %d -> %d)",
                    height, width, out_side);
    if (workspace_bytes < score_workspace_bytes(g, n))
        return fail(nullptr, TMAE_EINVAL, "workspace too small: %zu < %zu bytes", workspace_bytes, score_workspace_bytes(g, n));
    if (n > 0 && (reinterpret_cast<uintptr_t>(workspace) & 255) != 0)
        return fail(nullptr, TMAE_EINVAL, "workspace must be 256-byte aligned (histograms, tickets and the segmented image are carved out of it)");
    if (n > 65535) return fail(nullptr, TMAE_EINVAL, "at most 65535 images per call (got %d)", n);
    cudaError_t e = launch_generate_scores(gray, n, g, out->scores, out->s_map, out->t_map, out->segmented, workspace,
                                           reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "generate_scores: %s", cudaGetErrorString(e));
    return TMAE_OK;
}

// ---- engine self-tests ---------------------------------------------------------------------------------
static int engine_common(tmae_handle* tmp, const GemmDesc& d_in, int block_n, int impl, cudaStream_t st, int pair = 0) {
    GemmParams p;
    GemmDesc d = d_in;
    int reuse_bytes = 0;
    if (d.in_mode == IN_CONV) {          // same decision as add_gemm_group (block_n first, then whether the reuse stages fit)
        const int mt = (d.M + kBlockM - 1) / kBlockM;
        const int bn = block_n > 0 ? block_n : pick_block_n(mt, d.layer->Cout, 1);
        block_n = bn;
        reuse_bytes = conv_reuse_stage_bytes(tmp, d, bn, (d.layer->Cout + bn - 1) / bn, 1, pair != 0 && impl == 0);
        d.conv_reuse = reuse_bytes > 0;
    }
    int rc = fill_params(tmp, d, 1, &p, block_n);
    if (rc) return rc;
    GemmParams* dp = nullptr;
    if (cudaMalloc(reinterpret_cast<void**>(&dp), sizeof(GemmParams)) != cudaSuccess) return fail(tmp, TMAE_ENOMEM, "cudaMalloc params");
    // bring-up aid: TMAE_GEMM_TIMING=1 prints the per-phase globaltimer profile of the tensor-core kernel
    const bool timing = getenv("TMAE_GEMM_TIMING") != nullptr && impl == 0;
    __nv_bfloat16* bf16_out = nullptr;
    if (timing && getenv("TMAE_TIMING_BF16")) {      // time the bf16 same-row store path (persistent kernel for big grids); output discarded
        cudaMalloc(reinterpret_cast<void**>(&bf16_out), (size_t)p.M * p.N * 2);
        p.out[0].ptr = bf16_out; p.out[0].dtype = OUT_BF16; p.out[0].map = MAP_SAME; p.out[0].ld = p.N;
        if (getenv("TMAE_TIMING_GELU")) p.act = ACT_GELU;
    }
    const int ctas = ((p.M + kBlockM - 1) / kBlockM) * ((p.N + p.block_n - 1) / p.block_n);
    long long* dticks = nullptr;
    if (timing) {
        cudaMalloc(reinterpret_cast<void**>(&dticks), (size_t)ctas * 16 * sizeof(long long));
        cudaMemset(dticks, 0, (size_t)ctas * 16 * sizeof(long long));
        p.dbg_ticks = dticks;
    }
    cudaMemcpyAsync(dp, &p, sizeof(p), cudaMemcpyHostToDevice, st);
    if (pair && !p.pair_ok) { cudaFree(dp); return fail(tmp, TMAE_EINVAL, "pair launch needs a linear layer with block_n %% 32 == 0"); }
    if (pair == 2 && getenv("TMAE_GEMM_TIMING") != nullptr && impl == 0) {
        // bring-up aid for the persistent pair kernel: phase stamps of the first three tiles of every CTA
        long long* dt = nullptr;
        cudaMalloc(reinterpret_cast<void**>(&dt), (size_t)148 * 16 * sizeof(long long));
        cudaMemset(dt, 0, (size_t)148 * 16 * sizeof(long long));
        p.dbg_ticks = dt;
        cudaMemcpyAsync(dp, &p, sizeof(p), cudaMemcpyHostToDevice, st);
        gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), false, false, st, nullptr, 0, 0, 2);      // cold
        cudaStreamSynchronize(st);
        cudaEvent_t ev0, ev1; cudaEventCreate(&ev0); cudaEventCreate(&ev1);
        cudaEventRecord(ev0, st);
        cudaError_t e2 = gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), false, false, st, nullptr, 0, 0, 2);
        cudaEventRecord(ev1, st);
        cudaStreamSynchronize(st);
        float ms = 0; cudaEventElapsedTime(&ms, ev0, ev1);
        std::vector<long long> t((size_t)148 * 16);
        cudaMemcpy(t.data(), dt, t.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        double avg[16] = {0}; int nc = 0;
        for (int c = 0; c < 148; c += 2) if (t[c * 16]) { ++nc; for (int k = 1; k < 14; ++k) avg[k] += (double)(t[c * 16 + k] - t[c * 16]); }
        for (int k = 1; k < 14; ++k) avg[k] /= nc > 0 ? nc : 1;
        fprintf(stderr, "[pair-persistent timing] M=%d N=%d K=%d bn=%d leaders=%d | kernel %.1f us | ns since entry, tiles 0/1/2: mma_first %.0f/%.0f/%.0f  mma_last %.0f/%.0f/%.0f  "
                "accum_seen %.0f/%.0f/%.0f  epi_done %.0f/%.0f/%.0f | exit %.0f (%s)\n", p.M, p.N, p.b_kb_per_tap * 64, p.block_n, nc, ms * 1e3,
                avg[1], avg[5], avg[9], avg[2], avg[6], avg[10], avg[3], avg[7], avg[11], avg[4], avg[8], avg[12], avg[13], cudaGetErrorString(e2));
        p.dbg_ticks = nullptr;
        cudaMemcpyAsync(dp, &p, sizeof(p), cudaMemcpyHostToDevice, st);
        cudaStreamSynchronize(st);
        cudaFree(dt);
        // steady state, 50 launches back to back on the stream (PDL overlaps ramp and drain): the three bf16 store kernels
        for (int variant = 0; variant < 3; ++variant) {
            for (int i = 0; i < 3; ++i) gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), false, false, st, nullptr, 0, 0, variant);
            cudaStreamSynchronize(st);
            cudaEventRecord(ev0, st);
            for (int i = 0; i < 50; ++i) gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), false, false, st, nullptr, 0, 0, variant);
            cudaEventRecord(ev1, st);
            cudaStreamSynchronize(st);
            float msv = 0; cudaEventElapsedTime(&msv, ev0, ev1);
            fprintf(stderr, "[pair-persistent timing]   back-to-back x50, %s: %.2f us/launch = %.0f TFLOP/s\n",
                    variant == 0 ? "one CTA per tile / one-CTA persistent" : (variant == 1 ? "CTA pairs" : "persistent CTA pairs"),
                    msv * 1e3 / 50, 2.0 * p.M * p.N * p.b_kb_per_tap * 64 / (msv * 1e-3 / 50) / 1e12);
        }
    }
    cudaError_t e = gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), impl == 1, false, st, nullptr, 0, reuse_bytes, impl == 0 ? pair : 0);
    if (timing) {                      // second, warm launch is the one reported
        cudaStreamSynchronize(st);
        cudaEvent_t ev0, ev1; cudaEventCreate(&ev0); cudaEventCreate(&ev1);
        cudaEventRecord(ev0, st);
        e = gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), false, false, st, nullptr, 0, reuse_bytes);
        cudaEventRecord(ev1, st);
        cudaStreamSynchronize(st);
        float ms = 0; cudaEventElapsedTime(&ms, ev0, ev1);
        std::vector<long long> t((size_t)ctas * 16);
        cudaMemcpy(t.data(), dticks, t.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        long long tmin = t[0], tend = 0;
        for (int c = 0; c < ctas; ++c) { if (t[c * 16] < tmin) tmin = t[c * 16]; if (t[c * 16 + 6] > tend) tend = t[c * 16 + 6]; }
        double avg[16] = {0};
        for (int c = 0; c < ctas; ++c) for (int k = 1; k < 12; ++k) avg[k] += (double)(t[c * 16 + k] - t[c * 16]) / ctas;
        int smem = 0, kgroup = 1; const int stages = gemm_pick_stages(p.block_n, ctas, false, &smem, &kgroup);
        fprintf(stderr, "[gemm timing] M=%d N=%d Kb=%d taps=%d bn=%d ctas=%d stages=%d x%d smem=%d | kernel %.1f us (events), first-start..last-end %.1f us | "
                "per-CTA avg ns since entry: setup %.0f, tma0 %.0f, full0 %.0f, mma_done_issue %.0f, accum_seen %.0f, epi_done %.0f | first chunk: ldtm_done %.0f, staged %.0f, batch0 %.0f, batch1 %.0f\n",
                p.M, p.N, p.b_kb_per_tap, p.num_taps, p.block_n, ctas, stages, kgroup, smem, ms * 1e3,
                (tend - tmin) * 1e-3, avg[1], avg[2], avg[3], avg[4], avg[5], avg[6], avg[8], avg[9], avg[10], avg[11]);
        // steady-state cost of back-to-back dependent launches of this kernel: plain stream vs CUDA graph
        {
            p.dbg_ticks = nullptr;
            cudaMemcpyAsync(dp, &p, sizeof(p), cudaMemcpyHostToDevice, st);
            const int reps = 50;
            cudaStreamSynchronize(st);
            cudaEventRecord(ev0, st);
            for (int i = 0; i < reps; ++i) gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), false, false, st, nullptr, 0, reuse_bytes);
            cudaEventRecord(ev1, st);
            cudaStreamSynchronize(st);
            float ms_plain = 0; cudaEventElapsedTime(&ms_plain, ev0, ev1);
            cudaStream_t cs; cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
            cudaGraph_t graph = nullptr; cudaGraphExec_t gexec = nullptr;
            cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
            for (int i = 0; i < reps; ++i) gemm_launch(dp, 1, p.M, p.N, p.block_n, p.act, gemm_epi_kind(p), false, false, cs, nullptr, 0, reuse_bytes);
            cudaStreamEndCapture(cs, &graph);
            float ms_graph = -1;
            if (graph && cudaGraphInstantiate(&gexec, graph, 0) == cudaSuccess) {
                cudaGraphLaunch(gexec, cs); cudaStreamSynchronize(cs);
                cudaEventRecord(ev0, cs); cudaGraphLaunch(gexec, cs); cudaEventRecord(ev1, cs);
                cudaStreamSynchronize(cs);
                cudaEventElapsedTime(&ms_graph, ev0, ev1);
                cudaGraphExecDestroy(gexec);
            }
            if (graph) cudaGraphDestroy(graph);
            cudaStreamDestroy(cs);
            fprintf(stderr, "[gemm timing]   back-to-back x%d: %.2f us/launch (stream), %.2f us/launch (graph)\n", reps,
                    ms_plain * 1e3 / reps, ms_graph * 1e3 / reps);
        }
        if (bf16_out) {
            double a2[16] = {0};
            const int pc = ctas < 148 ? ctas : 148;
            for (int c = 0; c < pc; ++c) for (int k = 1; k < 13; ++k) a2[k] += (double)(t[c * 16 + k] - t[c * 16]) / pc;
            fprintf(stderr, "[gemm timing]   persistent tiles (ns since CTA entry): t0 mma %.0f-%.0f epi %.0f-%.0f | t1 mma %.0f-%.0f epi %.0f-%.0f | t2 mma %.0f-%.0f epi %.0f-%.0f\n",
                    a2[1], a2[2], a2[3], a2[4], a2[5], a2[6], a2[7], a2[8], a2[9], a2[10], a2[11], a2[12]);
            cudaFree(bf16_out);
        }
        cudaFree(dticks);
        cudaEventDestroy(ev0); cudaEventDestroy(ev1);
    }
    cudaError_t e2 = cudaStreamSynchronize(st);
    cudaFree(dp);
    if (e != cudaSuccess || e2 != cudaSuccess)
        return fail(tmp, TMAE_ECUDA, "engine launch: %s / %s", cudaGetErrorString(e), cudaGetErrorString(e2));
    return TMAE_OK;
}

static int make_tmp_handle(std::unique_ptr<tmae_handle>& tmp) {
    tmp.reset(new tmae_handle());
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return fail(nullptr, TMAE_ECUDA, "cuTensorMapEncodeTiled unavailable");
    tmp->encode = reinterpret_cast<PFN_encodeTiled>(fn);
    e = gemm_tc_configure();
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "gemm configure: %s", cudaGetErrorString(e));
    return TMAE_OK;
}

int tmae_gemm_bf16(const void* A, const void* B, const float* bias, float* Cmat, int M, int N, int K, int block_n,
                   int impl, void* stream) {
    if (!A || !B || !Cmat || M <= 0 || N <= 0 || K <= 0 || K % 8 != 0 || N % 8 != 0)
        return fail(nullptr, TMAE_EINVAL, "tmae_gemm_bf16: invalid shape (need K %% 8 == 0, N %% 8 == 0)");
    std::unique_ptr<tmae_handle> tmp;
    int rc = make_tmp_handle(tmp);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    // pack B [N, K] bf16 into [N, pad64(K)] (zero padded) and a zero bias if none
    const int Kp = pad64(K);
    __nv_bfloat16* wp = nullptr;
    float* bz = nullptr;
    std::vector<void*> pool;
    if ((rc = dev_alloc(tmp.get(), pool, &wp, (size_t)N * Kp)) || (rc = dev_alloc(tmp.get(), pool, &bz, (size_t)N))) {
        g_create_error = tmp->err; free_pool(pool); return rc;
    }
    cudaMemcpy2DAsync(wp, (size_t)Kp * 2, B, (size_t)K * 2, (size_t)K * 2, N, cudaMemcpyDeviceToDevice, st);
    if (bias) cudaMemcpyAsync(bz, bias, (size_t)N * 4, cudaMemcpyDeviceToDevice, st);
    Layer L;
    L.w = wp; L.bias = bz; L.Cout = N; L.Cin = K; L.taps = 1; L.nseg = 1; L.segc[0] = K; L.Kp = Kp; L.kb_tap = Kp / 64;
    GemmDesc d;
    d.layer = &L;
    d.seg[0] = seg(reinterpret_cast<const __nv_bfloat16*>(A), K, K);
    d.a_rows = M; d.M = M;
    d.out0 = outspec(Cmat, N, OUT_F32, MAP_SAME);
    rc = engine_common(tmp.get(), d, block_n, impl, st);
    if (rc) g_create_error = tmp->err;
    free_pool(pool);
    return rc;
}

// C (bf16) = act(A B^T + bias): the bf16 same-row store phases (TMA-store epilogue when block_n % 32 == 0).  variant 0 = one
// tile per CTA (or the one-CTA persistent kernel when the grid has more than two tiles per SM), 1 = CTA pairs, 2 = persistent
// CTA pairs, 3 = CUDA-core checker.
int tmae_gemm_bf16_out(const void* A, const void* B, const float* bias, void* Cmat, int M, int N, int K, int block_n, int gelu,
                       int variant, void* stream) {
    if (!A || !B || !Cmat || M <= 0 || N <= 0 || K <= 0 || K % 8 != 0 || N % 8 != 0 || variant < 0 || variant > 3)
        return fail(nullptr, TMAE_EINVAL, "tmae_gemm_bf16_out: invalid argument (need K %% 8 == 0, N %% 8 == 0, variant 0..3)");
    std::unique_ptr<tmae_handle> tmp;
    int rc = make_tmp_handle(tmp);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int Kp = pad64(K);
    __nv_bfloat16* wp = nullptr;
    float* bz = nullptr;
    std::vector<void*> pool;
    if ((rc = dev_alloc(tmp.get(), pool, &wp, (size_t)N * Kp)) || (rc = dev_alloc(tmp.get(), pool, &bz, (size_t)N))) {
        g_create_error = tmp->err; free_pool(pool); return rc;
    }
    cudaMemcpy2DAsync(wp, (size_t)Kp * 2, B, (size_t)K * 2, (size_t)K * 2, N, cudaMemcpyDeviceToDevice, st);
    if (bias) cudaMemcpyAsync(bz, bias, (size_t)N * 4, cudaMemcpyDeviceToDevice, st);
    Layer L;
    L.w = wp; L.bias = bz; L.Cout = N; L.Cin = K; L.taps = 1; L.nseg = 1; L.segc[0] = K; L.Kp = Kp; L.kb_tap = Kp / 64;
    GemmDesc d;
    d.layer = &L;
    d.seg[0] = seg(reinterpret_cast<const __nv_bfloat16*>(A), K, K);
    d.a_rows = M; d.M = M;
    d.act = gelu ? ACT_GELU : ACT_NONE;
    d.out0 = outspec(Cmat, N, OUT_BF16, MAP_SAME);
    rc = engine_common(tmp.get(), d, block_n, variant == 3 ? 1 : 0, st, variant == 3 ? 0 : variant);
    if (rc) g_create_error = tmp->err;
    free_pool(pool);
    return rc;
}

int tmae_conv3x3_bf16(const void* x, const float* wgt, const float* bias, float* out, int N, int s, int Cin, int Cout,
                      int gelu, int impl, void* stream) {
    if (!x || !wgt || !out || N <= 0 || s <= 0 || Cin % 8 != 0 || Cout % 8 != 0)
        return fail(nullptr, TMAE_EINVAL, "tmae_conv3x3_bf16: invalid shape");
    std::unique_ptr<tmae_handle> tmp;
    int rc = make_tmp_handle(tmp);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int Kp = pad64(Cin) * 9;
    std::vector<void*> pool;
    __nv_bfloat16* wp = nullptr;
    float* bz = nullptr;
    if ((rc = dev_alloc(tmp.get(), pool, &wp, (size_t)Cout * Kp)) || (rc = dev_alloc(tmp.get(), pool, &bz, (size_t)Cout))) {
        g_create_error = tmp->err; free_pool(pool); return rc;
    }
    int sg[1] = {Cin};
    cudaError_t e = launch_prepack_weight(wgt, wp, Cout, Cin, 9, 1, sg, 0, 1, st);
    if (bias) cudaMemcpyAsync(bz, bias, (size_t)Cout * 4, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { free_pool(pool); return fail(nullptr, TMAE_ECUDA, "conv3x3 staging: %s", cudaGetErrorString(e)); }
    Layer L;
    L.w = wp; L.bias = bz; L.Cout = Cout; L.Cin = Cin; L.taps = 9; L.nseg = 1; L.segc[0] = Cin; L.Kp = Kp; L.kb_tap = pad64(Cin) / 64;
    ConvGeom cg;
    if (!conv_geom(s, N, &cg)) { free_pool(pool); return fail(nullptr, TMAE_EINVAL, "tmae_conv3x3_bf16: grid side %d unsupported (1..128)", s); }
    GemmDesc d;
    d.layer = &L;
    d.seg[0] = seg(reinterpret_cast<const __nv_bfloat16*>(x), Cin, Cin);      // compact NHWC, read in place by 4-D TMA boxes
    d.a_rows = (long long)N * s * s; d.M = cg.m_tiles * kBlockM; d.in_mode = IN_CONV; d.side = s; d.n_img = N;
    d.act = gelu ? ACT_GELU : ACT_NONE;
    d.out0 = outspec(out, Cout, OUT_F32, MAP_SAME);
    rc = engine_common(tmp.get(), d, 0, impl == 2 ? 0 : impl, st, impl == 2);      // impl 2: CTA-pair (cta_group::2) launch
    if (rc) g_create_error = tmp->err;
    free_pool(pool);
    return rc;
}

// softmax(q k^T / sqrt(64)) v for qkv bf16 [N*T, 3C] (columns [3][H][64]) -> out bf16 [N*T, C]: the attention kernels of the
// encoder blocks stand-alone.  impl 0 = mma.sync kernel, 1 = tcgen05 / TMEM kernel (T <= 192).
int tmae_attention_bf16(const void* qkv, void* out, int N, int T, int H, int impl, void* stream) {
    if (!qkv || !out || N <= 0 || T <= 0 || H <= 0) return fail(nullptr, TMAE_EINVAL, "tmae_attention_bf16: invalid argument");
    std::unique_ptr<tmae_handle> tmp;
    int rc = make_tmp_handle(tmp);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int C = H * 64;
    cudaError_t e = attention_configure(T);
    if (e != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "attention configure: %s", cudaGetErrorString(e));
    if (impl >= 1 && impl <= 3) {          // 2 = the multi-stream ("lite") form of the tcgen05 kernel for short rows, 3 = duo (T = 65)
        if (!attention_tc_supported(T)) return fail(nullptr, TMAE_EINVAL, "tcgen05 attention needs T <= 384");
        CUtensorMap mq, mk;
        if ((rc = make_attention_maps(tmp.get(), reinterpret_cast<const __nv_bfloat16*>(qkv), (long long)N * T, C, T, impl, &mq, &mk))) {
            g_create_error = tmp->err; return rc;
        }
        long long* dbg = nullptr;
        const bool timing = getenv("TMAE_ATTN_TIMING") != nullptr;      // bring-up aid: per-phase clock64 stamps of CTA 0
        if (timing) { cudaMalloc(reinterpret_cast<void**>(&dbg), 64 * 16 * 8); cudaMemset(dbg, 0, 64 * 16 * 8); }
        e = launch_attention_tc(&mq, &mk, reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), N, T, H, C, 0.125f, st,
                                dbg, impl);
        if (timing) {
            cudaStreamSynchronize(st);
            std::vector<long long> hd(64 * 16);
            cudaMemcpy(hd.data(), dbg, hd.size() * 8, cudaMemcpyDeviceToHost);
            cudaFree(dbg);
            long long t0 = 0;
            for (int k = 0; k < 64 && hd[k * 16 + 5]; ++k) {
                if (k == 0) t0 = hd[0];
                fprintf(stderr, "[attn item %2d] mma: full %6lld S_issued %6lld p_ready %6lld PV_issued %6lld | wg: enter %6lld s_ready %6lld ld %6lld exp_done %6lld arrived %6lld o_ready %6lld o_ld %6lld stored %6lld\n",
                        k, hd[k * 16 + 0] - t0, hd[k * 16 + 1] - t0, hd[k * 16 + 2] - t0, hd[k * 16 + 3] - t0, hd[k * 16 + 4] - t0, hd[k * 16 + 5] - t0,
                        hd[k * 16 + 6] - t0, hd[k * 16 + 7] - t0, hd[k * 16 + 8] - t0, hd[k * 16 + 9] - t0, hd[k * 16 + 10] - t0, hd[k * 16 + 11] - t0);
            }
        }
    } else {
        e = launch_attention(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), N, T, H, C, 0.125f, st);
    }
    cudaError_t e2 = cudaStreamSynchronize(st);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "attention launch: %s / %s", cudaGetErrorString(e), cudaGetErrorString(e2));
    return TMAE_OK;
}

// softmax(q k^T / sqrt(32)) v for qkv bf16 [N*T, 3*H*32] (columns [3][H][32]) -> out bf16 [N*T, H*32]: the attention kernel of the
// synthesis plan's decoder blocks stand-alone.
int tmae_attention_hd32_bf16(const void* qkv, void* out, int N, int T, int H, void* stream) {
    if (!qkv || !out || N <= 0 || T <= 0 || H <= 0) return fail(nullptr, TMAE_EINVAL, "tmae_attention_hd32_bf16: invalid argument");
    if (!attention_hd32_supported(T)) return fail(nullptr, TMAE_EINVAL, "tmae_attention_hd32_bf16: T = %d does not fit shared memory", T);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cudaError_t e = launch_attention_hd32(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), N, T, H,
                                          1.0f / sqrtf(32.0f), st);
    cudaError_t e2 = cudaStreamSynchronize(st);
    if (e != cudaSuccess || e2 != cudaSuccess) return fail(nullptr, TMAE_ECUDA, "attention launch: %s / %s", cudaGetErrorString(e), cudaGetErrorString(e2));
    return TMAE_OK;
}

// x_out = resid + A B^T + bias (fp32 in / out, bf16 operands): the encoder's proj / fc2 epilogue.  pair = 1 runs the CTA-pair
// (cta_group::2) kernel, 0 the one-CTA kernel, impl 1 the CUDA-core checker.
int tmae_gemm_bf16_resid(const void* A, const void* B, const float* bias, const float* resid, float* Cmat, int M, int N, int K,
                         int block_n, int pair, int impl, void* stream) {
    if (!A || !B || !Cmat || !resid || M <= 0 || N <= 0 || K <= 0 || K % 8 != 0 || N % 8 != 0)
        return fail(nullptr, TMAE_EINVAL, "tmae_gemm_bf16_resid: invalid shape (need K %% 8 == 0, N %% 8 == 0)");
    std::unique_ptr<tmae_handle> tmp;
    int rc = make_tmp_handle(tmp);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int Kp = pad64(K);
    __nv_bfloat16* wp = nullptr;
    float* bz = nullptr;
    std::vector<void*> pool;
    if ((rc = dev_alloc(tmp.get(), pool, &wp, (size_t)N * Kp)) || (rc = dev_alloc(tmp.get(), pool, &bz, (size_t)N))) {
        g_create_error = tmp->err; free_pool(pool); return rc;
    }
    cudaMemcpy2DAsync(wp, (size_t)Kp * 2, B, (size_t)K * 2, (size_t)K * 2, N, cudaMemcpyDeviceToDevice, st);
    if (bias) cudaMemcpyAsync(bz, bias, (size_t)N * 4, cudaMemcpyDeviceToDevice, st);
    Layer L;
    L.w = wp; L.bias = bz; L.Cout = N; L.Cin = K; L.taps = 1; L.nseg = 1; L.segc[0] = K; L.Kp = Kp; L.kb_tap = Kp / 64;
    GemmDesc d;
    d.layer = &L;
    d.seg[0] = seg(reinterpret_cast<const __nv_bfloat16*>(A), K, K);
    d.a_rows = M; d.M = M;
    d.resid = resid; d.resid_ld = N; d.resid_map = MAP_SAME;
    d.out0 = outspec(Cmat, N, OUT_F32, MAP_SAME);
    rc = engine_common(tmp.get(), d, block_n, impl, st, pair != 0);
    if (rc) g_create_error = tmp->err;
    free_pool(pool);
    return rc;
}

// Precise (split-bf16) engine self-tests: fp32 operands in, split into (hi, lo) bf16 planes here, three tensor-core
// terms per product - the configuration every TMAE_FLAG_PRECISE_* layer runs in.
int tmae_gemm_split(const float* A, const float* B, const float* bias, float* Cmat, int M, int N, int K, int block_n,
                    int planes, int impl, void* stream) {
    if (!A || !B || !Cmat || M <= 0 || N <= 0 || K <= 0 || K % 8 != 0 || N % 8 != 0 || (planes != 2 && planes != 3))
        return fail(nullptr, TMAE_EINVAL, "tmae_gemm_split: invalid shape (need K %% 8 == 0, N %% 8 == 0)");
    std::unique_ptr<tmae_handle> tmp;
    int rc = make_tmp_handle(tmp);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int Kp = pad64(K);
    __nv_bfloat16 *wp = nullptr, *ap = nullptr;
    float* bz = nullptr;
    std::vector<void*> pool;
    const size_t a_plane = ((size_t)M * K + 63) / 64 * 64;
    const long long a_lo = planes == 2 ? (long long)a_plane : -(long long)a_plane;
    if ((rc = dev_alloc(tmp.get(), pool, &wp, (size_t)N * Kp * planes)) || (rc = dev_alloc(tmp.get(), pool, &bz, (size_t)N)) ||
        (rc = dev_alloc(tmp.get(), pool, &ap, a_plane * planes))) {
        g_create_error = tmp->err; free_pool(pool); return rc;
    }
    int sg[1] = {K};
    cudaError_t e = launch_prepack_weight(B, wp, N, K, 1, 1, sg, 0, planes, st);
    if (e == cudaSuccess) e = launch_f32_to_bf16(A, ap, (long long)M * K, a_lo, st);
    if (bias) cudaMemcpyAsync(bz, bias, (size_t)N * 4, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { free_pool(pool); return fail(nullptr, TMAE_ECUDA, "gemm_split staging: %s", cudaGetErrorString(e)); }
    Layer L;
    L.w = wp; L.bias = bz; L.Cout = N; L.Cin = K; L.taps = 1; L.nseg = 1; L.segc[0] = K; L.planes = planes; L.kb_tap = Kp / 64; L.Kp = Kp * planes;
    GemmDesc d;
    d.layer = &L;
    d.seg[0] = seg(ap, K, K, a_lo);
    d.a_rows = M; d.M = M;
    d.out0 = outspec(Cmat, N, OUT_F32, MAP_SAME);
    rc = engine_common(tmp.get(), d, block_n, impl, st);
    if (rc) g_create_error = tmp->err;
    free_pool(pool);
    return rc;
}

int tmae_conv3x3_split(const float* x, const float* wgt, const float* bias, float* out, int N, int s, int Cin, int Cout,
                       int gelu, int planes, int impl, void* stream) {
    if (!x || !wgt || !out || N <= 0 || s <= 0 || Cin % 8 != 0 || Cout % 8 != 0 || (planes != 2 && planes != 3))
        return fail(nullptr, TMAE_EINVAL, "tmae_conv3x3_split: invalid shape");
    std::unique_ptr<tmae_handle> tmp;
    int rc = make_tmp_handle(tmp);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int kp_tap = pad64(Cin);
    std::vector<void*> pool;
    __nv_bfloat16 *wp = nullptr, *xp = nullptr;
    float* bz = nullptr;
    const size_t x_plane = ((size_t)N * s * s * Cin + 63) / 64 * 64;
    const long long x_lo = planes == 2 ? (long long)x_plane : -(long long)x_plane;
    if ((rc = dev_alloc(tmp.get(), pool, &wp, (size_t)Cout * kp_tap * 9 * planes)) || (rc = dev_alloc(tmp.get(), pool, &bz, (size_t)Cout)) ||
        (rc = dev_alloc(tmp.get(), pool, &xp, x_plane * planes))) {
        g_create_error = tmp->err; free_pool(pool); return rc;
    }
    int sg[1] = {Cin};
    cudaError_t e = launch_prepack_weight(wgt, wp, Cout, Cin, 9, 1, sg, 0, planes, st);
    if (e == cudaSuccess) e = launch_f32_to_bf16(x, xp, (long long)N * s * s * Cin, x_lo, st);
    if (bias) cudaMemcpyAsync(bz, bias, (size_t)Cout * 4, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { free_pool(pool); return fail(nullptr, TMAE_ECUDA, "conv3x3_split staging: %s", cudaGetErrorString(e)); }
    Layer L;
    L.w = wp; L.bias = bz; L.Cout = Cout; L.Cin = Cin; L.taps = 9; L.nseg = 1; L.segc[0] = Cin; L.planes = planes; L.kb_tap = kp_tap / 64;
    L.Kp = kp_tap * 9 * planes;
    ConvGeom cg;
    if (!conv_geom(s, N, &cg)) { free_pool(pool); return fail(nullptr, TMAE_EINVAL, "tmae_conv3x3_split: grid side %d unsupported (1..128)", s); }
    GemmDesc d;
    d.layer = &L;
    d.seg[0] = seg(xp, Cin, Cin, x_lo);
    d.a_rows = (long long)N * s * s; d.M = cg.m_tiles * kBlockM; d.in_mode = IN_CONV; d.side = s; d.n_img = N;
    d.act = gelu ? ACT_GELU : ACT_NONE;
    d.out0 = outspec(out, Cout, OUT_F32, MAP_SAME);
    rc = engine_common(tmp.get(), d, 0, impl, st);
    if (rc) g_create_error = tmp->err;
    free_pool(pool);
    return rc;
}

// ---- profiling -----------------------------------------------------------------------------------------
int tmae_profile_enable(tmae_handle* h, int enable) {
    if (!h) return TMAE_EINVAL;
    h->profiling = enable != 0;
    h->prof_by_run = enable == 2;
    h->prof_used = 0;
    return TMAE_OK;
}

int tmae_profile_read(tmae_handle* h, tmae_profile_entry* entries, int max_entries, int* n_entries) {
    if (!h || !entries || !n_entries) return TMAE_EINVAL;
    tmae_profile_entry fam[FAM_COUNT];
    memset(fam, 0, sizeof(fam));
    for (int f = 0; f < FAM_COUNT; ++f) snprintf(fam[f].name, sizeof(fam[f].name), "%s", kFamilyNames[f]);
    for (size_t i = 0; i < h->prof_used; ++i) {
        const ProfRecord& r = h->prof[i];
        float ms = 0.f;
        cudaError_t e = cudaEventElapsedTime(&ms, r.begin, r.end);
        if (e != cudaSuccess) return fail(h, TMAE_ECUDA, "cudaEventElapsedTime: %s (synchronise the stream first)", cudaGetErrorString(e));
        tmae_profile_entry& f = fam[r.family];
        f.launches += r.launches;
        f.ms += ms;
        f.flops += r.flops;
        f.bytes += r.bytes;
        f.mma_flops += r.mma_flops;
    }
    int n = 0;
    for (int f = 0; f < FAM_COUNT && n < max_entries; ++f)
        if (fam[f].launches > 0) entries[n++] = fam[f];
    *n_entries = n;
    return TMAE_OK;
}

int tmae_profile_read_steps(tmae_handle* h, tmae_profile_step* steps, int max_steps, int* n_steps) {
    if (!h || !steps || !n_steps) return TMAE_EINVAL;
    int n = 0;
    for (size_t i = 0; i < h->prof_used && n < max_steps; ++i, ++n) {
        const ProfRecord& r = h->prof[i];
        float ms = 0.f;
        cudaError_t e = cudaEventElapsedTime(&ms, r.begin, r.end);
        if (e != cudaSuccess) return fail(h, TMAE_ECUDA, "cudaEventElapsedTime: %s (synchronise the stream first)", cudaGetErrorString(e));
        memset(&steps[n], 0, sizeof(steps[n]));
        snprintf(steps[n].name, sizeof(steps[n].name), "%s", r.tag.c_str());
        steps[n].ms = ms;
        steps[n].flops = r.flops;
        steps[n].ctas = r.ctas;
        steps[n].block_n = r.block_n;
    }
    *n_steps = n;
    return TMAE_OK;
}

}  // extern "C"
