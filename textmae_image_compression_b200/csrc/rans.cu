// rANS entropy coder of the codec's bitstream: compressai 1.2.4's format (BufferedRansEncoder.encode_with_indexes + flush,
// RansDecoder.decode_with_indexes over ryg_rans' rans64), restated in DESIGN.md section 7.
//   precision 16, 64-bit state, RANS64_L = 2^31, 32-bit words; escapes code the table's last symbol followed by 4-bit bypass
//   groups (a count as a run of 15s plus a remainder, then the raw value's nibbles, low nibble first).
// Encode: a parallel pass maps every (symbol, index) to its table entry plus the escape's raw value; a sequential pass per
// stream (one thread each) runs the reverse recurrence with precomputed reciprocals (no 64-bit division) and writes the
// words backwards into the stream's scratch region; a compaction pass packs the streams and writes their byte offsets.
// Decode: one warp per stream; the table set sits in shared memory, each symbol's CDF search is 32 probes per round with a
// ballot, indexes and words are read 32 at a time.  Every read of a stream is bounded by its length: words past the end
// read as 0 and set a status bit, so a truncated or corrupt stream decodes to garbage with a nonzero status, never out of
// bounds.
// Laned format (DESIGN.md section 7): a stream of W lanes is {W, byte length of every lane, the lanes}, lane l being the compressai
// stream of the symbols l, l + W, ...  The encode recurrence runs per (stream, lane) and a second compaction writes the header;
// the decode is one thread per (stream, lane), each with its own binary search and every read bounded by its lane.
#include <math.h>

#include <algorithm>
#include <map>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace tmae {

namespace {
constexpr uint64_t kRansL = 1ull << 31;
constexpr int kPrec = 16;
constexpr uint32_t kBypassMax = 15;              // (1 << 4) - 1
constexpr int kDecSmemMax = 200 * 1024;          // larger table sets stay in (L1-cached) global memory
constexpr unsigned kFull = 0xffffffffu;
}  // namespace

// ---- host: tables ------------------------------------------------------------------------------------------------
// compressai's pmf_to_quantized_cdf (cpp_exts/ops/ops.cpp) at precision 16: round p * 2^16 (in float, as the C++ does with
// its std::vector<float>), rescale by the total, partial sum with the last entry forced to 2^16, then give every empty bin
// one count stolen from the smallest bin with frequency > 1.
int pmf_to_quantized_cdf(const float* pmf, int n, int32_t* cdf_out) {
    if (!pmf || !cdf_out || n < 1) return TMAE_EINVAL;
    std::vector<uint32_t> cdf((size_t)n + 1);
    cdf[0] = 0;
    for (int i = 0; i < n; ++i) {
        const float p = pmf[i];
        if (!(p >= 0.f) || !isfinite(p) || p * 65536.f >= 4294967296.f) return TMAE_EINVAL;
        cdf[i + 1] = (uint32_t)roundf(p * (float)(1 << kPrec));
    }
    uint32_t total = 0;                          // std::accumulate(..., 0): int arithmetic, wraps like the original
    for (uint32_t v : cdf) total += v;
    if (total == 0) return TMAE_EINVAL;          // all-zero pmf: the original divides by zero
    for (auto& v : cdf) v = (uint32_t)(((1ull << kPrec) * v) / total);
    for (size_t i = 1; i < cdf.size(); ++i) cdf[i] += cdf[i - 1];
    cdf.back() = 1u << kPrec;
    for (int i = 0; i < (int)cdf.size() - 1; ++i) {
        if (cdf[i] != cdf[i + 1]) continue;
        uint32_t best_freq = ~0u;
        int best_steal = -1;
        for (int j = 0; j < (int)cdf.size() - 1; ++j) {
            const uint32_t f = cdf[j + 1] - cdf[j];
            if (f > 1 && f < best_freq) { best_freq = f; best_steal = j; }
        }
        if (best_steal < 0) return TMAE_EINVAL;  // more bins than counts
        if (best_steal < i) for (int j = best_steal + 1; j <= i; ++j) cdf[j]--;
        else for (int j = i + 1; j <= best_steal; ++j) cdf[j]++;
    }
    for (size_t i = 0; i < cdf.size(); ++i) cdf_out[i] = (int32_t)cdf[i];
    return TMAE_OK;
}

long long rans_bound_bytes(long long n) {
    // per symbol at most 1 put + 1 bypass-count put + 8 nibble puts (raw < 2^32), each emitting at most one word; + 2 flush words
    return n < 0 ? -1 : 4 * (10 * n + 2);
}

long long rans_bound_lanes_bytes(long long n, int lanes) {
    // the header, then per lane the bound of its ceil((n - l) / lanes) symbols: 4 (1 + lanes) + 4 (10 n + 2 lanes)
    return n < 0 || lanes < 1 || lanes > 32 ? -1 : 4 * (1 + lanes) + 4 * (10 * n + 2 * lanes);
}

namespace {
// ryg_rans' Rans64EncSymbolInit reciprocal: q = mulhi(x, rcp) >> shift == x / freq for x < 2^63 (freq >= 2)
void reciprocal(uint32_t freq, uint64_t* rcp, uint32_t* shift) {
    if (freq < 2) { *rcp = 0; *shift = 0; return; }
    uint32_t sh = 0;
    while (freq > (1u << sh)) sh++;
    uint64_t x0 = freq - 1, x1 = 1ull << (sh + 31);
    const uint64_t t1 = x1 / freq;
    x0 += (x1 % freq) << 32;
    const uint64_t t0 = x0 / freq;
    *rcp = t0 + (t1 << 32);
    *shift = sh - 1;
}
uint64_t host_div(uint64_t x, uint32_t freq, uint64_t rcp, uint32_t shift) {
    if (freq < 2) return x;
    return (uint64_t)(((unsigned __int128)x * rcp) >> 64) >> shift;
}
}  // namespace

void rans_free_tables(CdfTables* t) {
    if (t->cdf) cudaFree(t->cdf);
    if (t->enc) cudaFree(t->enc);
    *t = CdfTables();
}

int rans_build_tables(const int32_t* cdf, int n, int stride, const int32_t* len, const int32_t* off, CdfTables* out,
                      char* err, size_t err_len) {
    std::vector<int32_t> flat, meta((size_t)n * 3);
    for (int t = 0; t < n; ++t) {
        const int L = len[t];
        if (L < 3 || L > stride) { snprintf(err, err_len, "table %d: cdf length %d outside 3..%d", t, L, stride); return TMAE_EINVAL; }
        const int32_t* c = cdf + (size_t)t * stride;
        if (c[0] != 0 || c[L - 1] != (1 << kPrec)) { snprintf(err, err_len, "table %d: a cdf must start at 0 and end at 65536", t); return TMAE_EINVAL; }
        for (int i = 0; i + 1 < L; ++i)
            if (c[i + 1] <= c[i]) { snprintf(err, err_len, "table %d: cdf not strictly increasing at %d", t, i); return TMAE_EINVAL; }
        if (flat.size() + L > (size_t)1 << 30) { snprintf(err, err_len, "table set too large"); return TMAE_EINVAL; }
        meta[3 * t] = (int32_t)flat.size(); meta[3 * t + 1] = L; meta[3 * t + 2] = off[t];
        flat.insert(flat.end(), c, c + L);
    }
    // encoder entries: symbol v of table t at meta.start + v: {start | freq << 16, rcp shift, rcp lo, rcp hi}
    std::vector<uint4> enc(flat.size());
    std::map<uint32_t, std::pair<uint64_t, uint32_t>> rcps;
    for (int t = 0; t < n; ++t)
        for (int v = 0; v + 1 < meta[3 * t + 1]; ++v) {
            const int e = meta[3 * t] + v;
            const uint32_t start = (uint32_t)flat[e], freq = (uint32_t)(flat[e + 1] - flat[e]);   // 1..65535 (>= 2 bins)
            auto it = rcps.find(freq);
            if (it == rcps.end()) {
                uint64_t r; uint32_t s;
                reciprocal(freq, &r, &s);
                // the recurrence divides x in [x_max / 2^32, x_max) (after renormalisation) by freq: check the reciprocal
                // against the division at both ends and in between
                const uint64_t x_max = ((kRansL >> kPrec) << 32) * freq;
                const uint64_t probes[6] = {kRansL, kRansL + freq - 1, x_max - 1, x_max - freq, x_max / 3, (x_max >> 32) + 12345};
                for (uint64_t x : probes)
                    if (host_div(x, freq, r, s) != x / freq) { snprintf(err, err_len, "reciprocal of %u inexact", freq); return TMAE_EINVAL; }
                it = rcps.emplace(freq, std::make_pair(r, s)).first;
            }
            enc[e] = make_uint4(start | (freq << 16), it->second.second, (uint32_t)it->second.first, (uint32_t)(it->second.first >> 32));
        }
    CdfTables t;
    t.n = n;
    t.entries = (int)flat.size();
    cudaError_t e = cudaMalloc(&t.cdf, (flat.size() + meta.size()) * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMalloc(&t.enc, enc.size() * sizeof(uint4));
    if (e == cudaSuccess) e = cudaMemcpy(t.cdf, flat.data(), flat.size() * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(t.cdf + flat.size(), meta.data(), meta.size() * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(t.enc, enc.data(), enc.size() * sizeof(uint4), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        rans_free_tables(&t);
        snprintf(err, err_len, "cdf table upload: %s", cudaGetErrorString(e));
        return TMAE_ECUDA;
    }
    t.meta = t.cdf + flat.size();
    *out = t;
    return TMAE_OK;
}

// ---- encode ------------------------------------------------------------------------------------------------------
// Pass 1, thread per symbol: record = {table entry of the coded value, escape ? 0x80000000 | raw : 0}.
__global__ void __launch_bounds__(256)
rans_map_kernel(const int32_t* __restrict__ sym, const int32_t* __restrict__ idx, long long total, int n_per,
                const int* __restrict__ meta, int n_tab, uint2* __restrict__ rec, int32_t* __restrict__ status) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int t = idx[i];
    if (t < 0 || t >= n_tab) { atomicOr(status + i / n_per, RANS_ST_BAD_INDEX); t = 0; }
    const int start = meta[3 * t], max_value = meta[3 * t + 1] - 2;
    const long long value = (long long)sym[i] - meta[3 * t + 2];
    long long raw = -1;
    if (value < 0) raw = -2 * value - 1;
    else if (value >= max_value) raw = 2 * (value - max_value);
    if (raw >= (1ll << 31)) { atomicOr(status + i / n_per, RANS_ST_RANGE); raw = 0; }
    rec[i] = raw < 0 ? make_uint2((uint32_t)(start + value), 0u) : make_uint2((uint32_t)(start + max_value), 0x80000000u | (uint32_t)raw);
}

__device__ __forceinline__ void enc_emit(uint64_t& x, uint64_t x_max, uint32_t* base, long long& wp) {
    if (x >= x_max) { base[--wp] = (uint32_t)x; x >>= 32; }
}
__device__ __forceinline__ void enc_put_bits(uint64_t& x, uint32_t v, uint32_t* base, long long& wp) {
    enc_emit(x, (kRansL >> 4) << 32, base, wp);
    x = (x << 4) | v;
}

// Pass 2, thread per (stream, lane): the reverse recurrence from x = L over the lane's entries (entries lane, lane + lanes, ...
// of the stream), words written backwards from the end of region r = s * lanes + lane, [r * cap_words, (r + 1) * cap_words);
// then the two flush words (low word first).  lanes = 1: one chain per stream, compressai's format.
__global__ void __launch_bounds__(32)
rans_encode_kernel(const uint2* __restrict__ rec, const uint4* __restrict__ enc, int n_streams, int n_per, int lanes,
                   uint32_t* __restrict__ scratch, long long cap_words, long long* __restrict__ n_words) {
    const int rg = blockIdx.x * blockDim.x + threadIdx.x;
    if (rg >= n_streams * lanes) return;
    const int s = rg / lanes, lane = rg - s * lanes;
    uint32_t* base = scratch + (size_t)rg * cap_words;
    long long wp = cap_words;
    uint64_t x = kRansL;
    const uint2* r = rec + (size_t)s * n_per;
    for (int i = n_per > lane ? lane + (n_per - 1 - lane) / lanes * lanes : -1; i >= 0; i -= lanes) {
        const uint2 e = r[i];
        if (e.y) {
            const uint32_t raw = e.y & 0x7fffffffu;
            int nb = 0;
            while (nb < 8 && (raw >> (4 * nb)) != 0) ++nb;
            for (int j = nb - 1; j >= 0; --j) enc_put_bits(x, (raw >> (4 * j)) & kBypassMax, base, wp);
            enc_put_bits(x, (uint32_t)(nb % kBypassMax), base, wp);
            for (int k = nb / kBypassMax; k > 0; --k) enc_put_bits(x, kBypassMax, base, wp);
        }
        const uint4 q = __ldg(enc + e.x);
        const uint32_t start = q.x & 0xffffu, freq = q.x >> 16;
        enc_emit(x, ((kRansL >> kPrec) << 32) * freq, base, wp);
        const uint64_t rcp = ((uint64_t)q.w << 32) | q.z;
        const uint64_t d = freq < 2 ? x : (__umul64hi(x, rcp) >> q.y);
        x = (d << kPrec) + (x - d * freq) + start;
    }
    base[--wp] = (uint32_t)(x >> 32);
    base[--wp] = (uint32_t)x;
    n_words[rg] = cap_words - wp;
}

// sum of v[0, n) over a block of 256 threads
__device__ __forceinline__ long long block_sum256(const long long* __restrict__ v, long long n) {
    __shared__ long long part[8];
    long long acc = 0;
    for (long long j = threadIdx.x; j < n; j += blockDim.x) acc += v[j];
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    long long sum = 0;
    for (int w = 0; w < 8; ++w) sum += part[w];
    return sum;
}

// Pass 3, block per stream: byte offset = sum of the earlier streams' sizes; copy the words to the packed output.
__global__ void __launch_bounds__(256)
rans_compact_kernel(const uint32_t* __restrict__ scratch, long long cap_words, const long long* __restrict__ n_words, int n_streams,
                    uint8_t* __restrict__ out, long long capacity, int64_t* __restrict__ offsets, int32_t* __restrict__ status) {
    const int s = blockIdx.x;
    const long long off = block_sum256(n_words, s) * 4;
    const long long nw = n_words[s];
    if (threadIdx.x == 0) {
        offsets[s] = off;
        if (s == n_streams - 1) offsets[n_streams] = off + nw * 4;
        if (off + nw * 4 > capacity) atomicOr(status + s, RANS_ST_OVERFLOW);
    }
    if (off + nw * 4 > capacity) return;
    const uint32_t* src = scratch + (size_t)(s + 1) * cap_words - nw;
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + off);      // off is a multiple of 4
    for (long long j = threadIdx.x; j < nw; j += blockDim.x) dst[j] = src[j];
}

// Pass 3 of the laned format, block per stream: the stream is the words {lanes, byte length of every lane, the lanes in order};
// its byte offset is the sum of the earlier streams' sizes.
__global__ void __launch_bounds__(256)
rans_compact_lanes_kernel(const uint32_t* __restrict__ scratch, long long cap_words, const long long* __restrict__ n_words, int n_streams,
                          int lanes, uint8_t* __restrict__ out, long long capacity, int64_t* __restrict__ offsets,
                          int32_t* __restrict__ status) {
    const int s = blockIdx.x;
    const long long off = (block_sum256(n_words, (long long)s * lanes) + (long long)s * (1 + lanes)) * 4;
    const long long* nw = n_words + (size_t)s * lanes;
    long long total = 1 + lanes;
    for (int l = 0; l < lanes; ++l) total += nw[l];
    if (threadIdx.x == 0) {
        offsets[s] = off;
        if (s == n_streams - 1) offsets[n_streams] = off + total * 4;
        if (off + total * 4 > capacity) atomicOr(status + s, RANS_ST_OVERFLOW);
    }
    if (off + total * 4 > capacity) return;
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + off);
    if (threadIdx.x == 0) dst[0] = (uint32_t)lanes;
    if ((int)threadIdx.x < lanes) dst[1 + threadIdx.x] = (uint32_t)(nw[threadIdx.x] * 4);
    dst += 1 + lanes;
    for (int l = 0; l < lanes; ++l) {
        const uint32_t* src = scratch + ((size_t)s * lanes + l + 1) * cap_words - nw[l];
        for (long long j = threadIdx.x; j < nw[l]; j += blockDim.x) dst[j] = src[j];
        dst += nw[l];
    }
}

cudaError_t launch_rans_encode(const int32_t* sym, const int32_t* idx, int n_streams, int n_per, int lanes, const CdfTables& tab,
                               uint2* rec, uint32_t* scratch, long long cap_words, long long* n_words, uint8_t* out, long long capacity,
                               int64_t* offsets, int32_t* status, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(status, 0, sizeof(int32_t) * n_streams, st);
    if (e != cudaSuccess) return e;
    const long long total = (long long)n_streams * n_per;
    if (total > 0) {
        rans_map_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(sym, idx, total, n_per, tab.meta, tab.n, rec, status);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    const int chains = n_streams * std::max(lanes, 1);
    rans_encode_kernel<<<(chains + 31) / 32, 32, 0, st>>>(rec, tab.enc, n_streams, n_per, std::max(lanes, 1), scratch, cap_words, n_words);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (lanes == 0)
        rans_compact_kernel<<<n_streams, 256, 0, st>>>(scratch, cap_words, n_words, n_streams, out, capacity, offsets, status);
    else
        rans_compact_lanes_kernel<<<n_streams, 256, 0, st>>>(scratch, cap_words, n_words, n_streams, lanes, out, capacity, offsets, status);
    return cudaGetLastError();
}

// ---- decode ------------------------------------------------------------------------------------------------------
namespace {
// one stream's reader: a window of 32 words in the lanes' registers plus the next window already in flight, so the refill
// after every 32 words does not wait on a global load; every read bounded by the stream's length
struct WordReader {
    const uint32_t* w;
    unsigned n, base, pos;       // words, window start, next word
    uint32_t buf, nxt;           // words base + lane and base + 32 + lane
    int bad;
    __device__ __forceinline__ uint32_t fetch(unsigned j) const { return j < n ? __ldg(w + j) : 0u; }
    __device__ __forceinline__ void load(int lane) {     // base = pos rounded down to a window
        base = pos & ~31u;
        buf = fetch(base + lane);
        nxt = fetch(base + 32 + lane);
    }
    __device__ __forceinline__ uint32_t next(int lane) {
        if (pos - base >= 32) { base += 32; buf = nxt; nxt = fetch(base + 32 + lane); }   // pos advances by one word at a time
        const uint32_t v = __shfl_sync(kFull, buf, pos - base);
        if (pos >= n) bad |= RANS_ST_OVERRUN;
        ++pos;
        return v;
    }
};

// one lane's reader (laned format): words [pos, end) of the stream, the next word already in flight
struct LaneReader {
    const uint32_t* w;
    unsigned pos, end;
    uint32_t nxt;
    int bad;
    __device__ __forceinline__ uint32_t fetch(unsigned j) const { return j < end ? __ldg(w + j) : 0u; }
    __device__ __forceinline__ uint32_t next() {
        const uint32_t v = nxt;
        if (pos >= end) bad |= RANS_ST_OVERRUN;
        nxt = fetch(++pos);
        return v;
    }
};

// The table set, [cdf entries | meta 3 per table], staged in shared memory when a.use_smem (the tables are constant: staged
// while the predecessor finishes); then the per-call pointers, from the IoBlock in a decode-plan replay.
__device__ __forceinline__ const int* dec_prologue(const RansDecArgs& a, int* smem_tab, const uint8_t*& data, const int64_t*& offsets,
                                                   const int32_t*& indexes, int32_t*& status) {
    const int* tab = a.cdf;
    if (a.use_smem) {
        const int n_words_tab = a.entries + 3 * a.n_tab;
        for (int j = threadIdx.x; j < n_words_tab; j += blockDim.x) smem_tab[j] = __ldg(a.cdf + j);
        __syncthreads();
        tab = smem_tab;
    }
    pdl_wait();
    data = a.data;
    offsets = a.offsets;
    indexes = a.indexes;
    status = a.status;
    if (a.io) {
        const bool y = a.io_stream == 1;
        data = y ? a.io->y_data : a.io->z_data;
        offsets = y ? a.io->y_offsets : a.io->z_offsets;
        status = a.io->status;
        if (y) indexes = a.io->out.y_indexes;
    }
    return tab;
}

// Decodes past symbol sv = [start, start + freq) of a table of length L and renormalises; for the escape symbol (sv = L - 2) then
// the bypass count and the raw value's nibbles.  Returns the value before the table's offset.  next() yields the stream's next word.
template <class Next>
__device__ __forceinline__ int dec_symbol(uint64_t& x, int sv, int L, uint32_t start, uint32_t freq, Next&& next, int& bad) {
    x = freq * (x >> kPrec) + (x & 0xffff) - start;
    if (x < kRansL) x = (x << 32) | next();
    if (sv != L - 2) return sv;
    auto get4 = [&]() -> uint32_t {
        const uint32_t v = (uint32_t)(x & kBypassMax);
        x >>= 4;
        if (x < kRansL) x = (x << 32) | next();
        return v;
    };
    uint32_t v = get4();
    int nb = (int)v;
    while (v == kBypassMax && nb <= 8) { v = get4(); nb += (int)v; }
    if (nb > 8) { bad |= RANS_ST_MALFORMED; nb = 8; }      // our encoder never writes more than 8 nibbles
    uint32_t raw = 0;
    for (int j = 0; j < nb; ++j) raw |= get4() << (4 * j);
    const int r = (int)raw;                   // int32 arithmetic as compressai's decoder
    const int value = r >> 1;
    return (r & 1) ? -value - 1 : value + (L - 2);
}
}  // namespace

// Warp per stream: decodes symbols [a.begin, a.end) of every stream, continuing from (and leaving) the state in a.state unless
// a.init / a.fin.
__global__ void __launch_bounds__(256)
rans_decode_kernel(RansDecArgs a) {
    extern __shared__ int smem_tab[];
    const uint8_t* data;
    const int64_t* offsets;
    const int32_t* indexes;
    int32_t* status;
    const int* tab = dec_prologue(a, smem_tab, data, offsets, indexes, status);
    const int* meta = tab + a.entries;
    const int lane = threadIdx.x & 31;
    const int s = blockIdx.x * a.streams_per_block + (threadIdx.x >> 5);
    if ((int)(threadIdx.x >> 5) >= a.streams_per_block || s >= a.n_streams) return;

    // the stream: bytes [offsets[s], offsets[s + 1]) of data; a malformed range decodes nothing (reads as zeros)
    const long long b0 = offsets[s], b1 = offsets[s + 1];
    WordReader rd;
    rd.bad = 0;
    if (b0 < 0 || b1 < b0 || (b0 & 3) || ((b1 - b0) & 3) || (b1 - b0) / 4 > 0xffffffffll) {
        rd.bad = RANS_ST_MALFORMED;
        rd.w = reinterpret_cast<const uint32_t*>(data);
        rd.n = 0;
    } else {
        rd.w = reinterpret_cast<const uint32_t*>(data + b0);
        rd.n = (unsigned)((b1 - b0) / 4);
    }
    uint64_t x;
    if (a.init) {
        rd.pos = 0; rd.load(lane);
        const uint32_t lo = rd.next(lane), hi = rd.next(lane);
        x = ((uint64_t)hi << 32) | lo;
    } else {
        x = a.state[s].x;
        rd.pos = a.state[s].pos;
        rd.load(lane);
    }
    const int32_t* ix = indexes ? indexes + (size_t)s * a.idx_stride : nullptr;
    int32_t* out = a.symbols + (size_t)s * a.sym_stride;
    for (int i0 = a.begin; i0 < a.end; i0 += 32) {
        const int cnt = min(32, a.end - i0);
        int my_idx = 0;
        if (lane < cnt) my_idx = ix ? ix[i0 + lane] : (i0 + lane) / a.idx_div;
        int my_sym = 0;
        for (int k = 0; k < cnt; ++k) {
            int t = __shfl_sync(kFull, my_idx, k);
            if (t < 0 || t >= a.n_tab) { rd.bad |= RANS_ST_BAD_INDEX; t = 0; }
            const int ts = meta[3 * t], L = meta[3 * t + 1], offset = meta[3 * t + 2];
            const int* c = tab + ts;
            const int cf = (int)(x & 0xffff);
            // largest s in [0, L - 2] with c[s] <= cf (c[0] = 0 <= cf; c[L - 1] = 65536 > cf)
            int lo = 0, hi = L - 1;
            while (hi - lo > 32) {
                const int step = (hi - lo + 31) >> 5;
                const int p = lo + lane * step;
                const unsigned b = __ballot_sync(kFull, p < hi && c[p] <= cf);
                lo += (__popc(b) - 1) * step;
                hi = min(lo + step, hi);
            }
            const int p = lo + lane;
            const int sv = lo + __popc(__ballot_sync(kFull, p < hi && c[p] <= cf)) - 1;
            const uint32_t start = (uint32_t)c[sv], freq = (uint32_t)(c[sv + 1] - c[sv]);
            const int value = dec_symbol(x, sv, L, start, freq, [&]() { return rd.next(lane); }, rd.bad);
            if (lane == k) my_sym = value + offset;
        }
        if (lane < cnt) out[i0 + lane] = my_sym;
    }
    if (lane == 0) {
        int st = rd.bad;
        if (a.fin && (x != kRansL || rd.pos != rd.n)) st |= RANS_ST_UNFINISHED;
        if (a.init && a.status_reset) status[s] = st;
        else if (st) atomicOr(status + s, st);
        if (!a.fin) { a.state[s].x = x; a.state[s].pos = rd.pos; }
    }
}

// Laned format, thread per (stream, lane): lane l of a stream decodes its symbols l, l + lanes, ... within [a.begin, a.end), with
// its own binary search of the table; consecutive lanes read consecutive indexes and write consecutive symbols.  A block holds
// a.streams_per_block whole streams, whose status bits are gathered in shared memory.  State between stages: a.state[s * lanes
// + l] = {x, next word, end word}, word positions relative to the stream's first byte.
__global__ void __launch_bounds__(256)
rans_decode_lanes_kernel(RansDecArgs a) {
    extern __shared__ int smem_tab[];
    __shared__ int st_img[256];
    const uint8_t* data;
    const int64_t* offsets;
    const int32_t* indexes;
    int32_t* status;
    const int* tab = dec_prologue(a, smem_tab, data, offsets, indexes, status);
    const int* meta = tab + a.entries;
    const int W = a.lanes;
    const int j = threadIdx.x / W, l = threadIdx.x - j * W;
    const int s = blockIdx.x * a.streams_per_block + j;
    if ((int)threadIdx.x < a.streams_per_block) st_img[threadIdx.x] = 0;
    __syncthreads();
    if (j < a.streams_per_block && s < a.n_streams) {
        const long long b0 = offsets[s], b1 = offsets[s + 1];
        const bool range_ok = !(b0 < 0 || b1 < b0 || (b0 & 3) || ((b1 - b0) & 3) || (b1 - b0) / 4 > 0xffffffffll);
        LaneReader rd;
        rd.w = reinterpret_cast<const uint32_t*>(data + (range_ok ? b0 : 0));
        rd.bad = 0;
        uint64_t x;
        if (a.init) {
            // header: {W, byte length of every lane (a multiple of 4, >= 8)}, lengths adding up to the stream
            const unsigned n = range_ok ? (unsigned)((b1 - b0) / 4) : 0u;
            bool ok = range_ok && n >= 1u + W && __ldg(rd.w) == (unsigned)W;
            unsigned long long sum = 1 + W, begin = 0;
            for (int k = 0; ok && k < W; ++k) {
                const uint32_t len = __ldg(rd.w + 1 + k);
                if ((len & 3) || len < 8) ok = false;
                if (k == l) begin = sum;
                sum += len / 4;
            }
            if (ok && sum == n) {
                rd.pos = (unsigned)begin;
                rd.end = (unsigned)begin + __ldg(rd.w + 1 + l) / 4;
            } else {
                rd.bad = RANS_ST_MALFORMED;
                rd.pos = rd.end = 0;
            }
            rd.nxt = rd.fetch(rd.pos);
            const uint32_t lo = rd.next(), hi = rd.next();
            x = ((uint64_t)hi << 32) | lo;
        } else {
            const RansDecState q = a.state[(size_t)s * W + l];
            x = q.x; rd.pos = q.pos; rd.end = q.pad;
            rd.nxt = rd.fetch(rd.pos);
        }
        const int32_t* ix = indexes ? indexes + (size_t)s * a.idx_stride : nullptr;
        int32_t* out = a.symbols + (size_t)s * a.sym_stride;
        // the index loads take longer than a symbol's decode: kAhead of them stay in flight, each in a fixed register slot (the
        // loop body is unrolled over the slots, so no register move waits on a pending load)
        constexpr int kAhead = 4;
        auto index_at = [&](int k) { return k < a.end ? (ix ? ix[k] : k / a.idx_div) : 0; };
        int i = a.begin + ((l - a.begin) % W + W) % W;              // first symbol of this lane in [begin, end)
        int tq[kAhead];
#pragma unroll
        for (int k = 0; k < kAhead; ++k) tq[k] = index_at(i + k * W);
        for (; i < a.end; i += kAhead * W) {
#pragma unroll
            for (int k = 0; k < kAhead; ++k) {
                const int ik = i + k * W;
                if (ik >= a.end) break;
                int t = tq[k];
                tq[k] = index_at(ik + kAhead * W);
                if (t < 0 || t >= a.n_tab) { rd.bad |= RANS_ST_BAD_INDEX; t = 0; }
                const int ts = meta[3 * t], L = meta[3 * t + 1], offset = meta[3 * t + 2];
                const int* c = tab + ts;
                const int cf = (int)(x & 0xffff);
                int lo = 0, hi = L - 1;                              // c[lo] <= cf < c[hi]
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (c[mid] <= cf) lo = mid; else hi = mid;
                }
                const uint32_t start = (uint32_t)c[lo], freq = (uint32_t)(c[lo + 1] - c[lo]);
                int esc_bad = 0;         // not rd.bad itself: aliasing the reader's member makes ptxas keep it on the stack
                out[ik] = dec_symbol(x, lo, L, start, freq, [&]() { return rd.next(); }, esc_bad) + offset;
                rd.bad |= esc_bad;
            }
        }
        int stv = rd.bad;
        if (a.fin && (x != kRansL || rd.pos != rd.end)) stv |= RANS_ST_UNFINISHED;
        if (!a.fin) { RansDecState q; q.x = x; q.pos = rd.pos; q.pad = rd.end; a.state[(size_t)s * W + l] = q; }
        if (stv) atomicOr(st_img + j, stv);
    }
    __syncthreads();
    const int si = blockIdx.x * a.streams_per_block + threadIdx.x;
    if ((int)threadIdx.x < a.streams_per_block && si < a.n_streams) {
        const int v = st_img[threadIdx.x];
        if (a.init && a.status_reset) status[si] = v;
        else if (v) atomicOr(status + si, v);
    }
}

cudaError_t launch_rans_decode(RansDecArgs a, cudaStream_t st) {
    if (a.n_streams <= 0) return cudaSuccess;
    const size_t tab_bytes = (size_t)(a.entries + 3 * a.n_tab) * 4;
    a.use_smem = tab_bytes <= (size_t)kDecSmemMax;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(rans_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDecSmemMax);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(rans_decode_lanes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDecSmemMax);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    // spread the streams over the SMs (every warp's / thread's loop is latency-bound)
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const int spread = std::max(1, (a.n_streams + sms - 1) / sms);
    if (a.lanes > 0) {           // whole streams per block; 256 threads however few lanes, so that the table staging is as fast
        a.streams_per_block = std::min(256 / a.lanes, spread);      // as the warp kernel's
        const int blocks = (a.n_streams + a.streams_per_block - 1) / a.streams_per_block;
        return launch_k(rans_decode_lanes_kernel, dim3(blocks), dim3(256), a.use_smem ? tab_bytes : 0, st, true, a);
    }
    a.streams_per_block = std::min(8, spread);     // warp per stream, at most 8 per block
    const int blocks = (a.n_streams + a.streams_per_block - 1) / a.streams_per_block;
    return launch_k(rans_decode_kernel, dim3(blocks), dim3(256), a.use_smem ? tab_bytes : 0, st, true, a);
}

}  // namespace tmae
