// Image containers (DESIGN.md section 7): one self-contained byte string per image.  Little-endian 32-bit words:
//   0 magic "TMAE" | 1 version, accuracy mode, W_y, W_z (a byte each) | 2 img_size (16 bits), patch_size (8), reserved (8)
//   | 3 K (16 bits), reserved (16) | 4 model tag | 5 z stream bytes | 6 y stream bytes
//   | ids_keep[0..K) in w = max(1, bit_length(L - 1)) bits each, LSB-first, zero-padded to a word | z stream | y stream
// Pack: one CTA per image after the two rANS encodes; the container's offset is the sum of the earlier containers' lengths,
// which the encodes' stream offsets (exclusive prefix sums) already give (for the tiles of pictures, plus the picture headers).  Parse: one CTA per container, the first stage of the
// decode; it validates the container against the handle and hands the decoders the byte ranges of the two streams (empty for a
// container it refuses, so nothing outside a container is ever read).
#include "common.cuh"
#include "kernels.h"

namespace tmae {

namespace {
constexpr int kHeaderWords = 7;

// bits [32 i, 32 i + 32) of the packed ids (LSB-first)
__device__ __forceinline__ uint32_t pack_id_word(const int64_t* ids, int K, int w, int i) {
    uint32_t v = 0;
    const long long b0 = 32ll * i;
    for (long long j = b0 / w; j < K && j * w < b0 + 32; ++j) {
        const uint32_t id = (uint32_t)ids[j];
        const long long sh = j * w - b0;
        v |= sh >= 0 ? id << sh : id >> -sh;
    }
    return v;
}

// id j of the packed ids starting at word pointer p (the section's words all lie inside the container)
__device__ __forceinline__ uint32_t unpack_id(const uint32_t* p, int w, int j) {
    const long long b = (long long)j * w;
    const int sh = (int)(b & 31);
    const uint32_t* q = p + (b >> 5);
    uint32_t v = __ldg(q) >> sh;
    if (sh + w > 32) v |= __ldg(q + 1) << (32 - sh);
    return w == 32 ? v : v & ((1u << w) - 1);
}
}  // namespace

// Byte offset and length of container n in the output: the containers before it back to back, plus (pictures) the header and
// length table of its picture and of every picture before it.
__device__ __forceinline__ void image_extent(const int64_t* y_off, const int64_t* z_off, long long fixed, int T, int n,
                                             long long* off, long long* len) {
    const long long gap = T ? (long long)(n / T + 1) * 4 * (4 + T) : 0;
    *off = n * fixed + (y_off[n] - y_off[0]) + (z_off[n] - z_off[0]) + gap;
    *len = fixed + (y_off[n + 1] - y_off[n]) + (z_off[n + 1] - z_off[n]);
}

__global__ void __launch_bounds__(256)
image_pack_kernel(const int64_t* __restrict__ ids_keep, const uint8_t* __restrict__ y_bytes, const int64_t* __restrict__ y_off,
                  const int32_t* __restrict__ y_st, const uint8_t* __restrict__ z_bytes, const int64_t* __restrict__ z_off,
                  const int32_t* __restrict__ z_st, ImageFields f, int N, uint8_t* __restrict__ out, long long capacity,
                  int64_t* __restrict__ offsets, int32_t* __restrict__ status, PictureGroup g) {
    const int n = blockIdx.x;
    const int id_words = (int)(((long long)f.K * f.id_bits + 31) / 32);
    const long long fixed = 4ll * (kHeaderWords + id_words);
    long long off, len;
    image_extent(y_off, z_off, fixed, g.T, n, &off, &len);
    const long long y_len = y_off[n + 1] - y_off[n], z_len = z_off[n + 1] - z_off[n];
    const bool fits = off + len <= capacity;
    if (threadIdx.x == 0) {
        offsets[n] = off;
        if (n == N - 1) offsets[N] = off + len;
        status[n] = y_st[n] | z_st[n] | (fits ? 0 : RANS_ST_OVERFLOW);
    }
    if (fits) {
        uint32_t* dst = reinterpret_cast<uint32_t*>(out + off);       // off, the header and every section: multiples of 4
        if (threadIdx.x == 0) {
            dst[0] = kImageMagic; dst[1] = f.word1; dst[2] = f.word2; dst[3] = f.word3; dst[4] = f.tag;
            dst[5] = (uint32_t)z_len; dst[6] = (uint32_t)y_len;
        }
        const int64_t* ids = ids_keep + (size_t)n * f.K;
        for (int i = threadIdx.x; i < id_words; i += blockDim.x) dst[kHeaderWords + i] = pack_id_word(ids, f.K, f.id_bits, i);
        dst += kHeaderWords + id_words;
        const uint32_t* zs = reinterpret_cast<const uint32_t*>(z_bytes + z_off[n]);
        for (long long i = threadIdx.x; i < z_len / 4; i += blockDim.x) dst[i] = zs[i];
        dst += z_len / 4;
        const uint32_t* ys = reinterpret_cast<const uint32_t*>(y_bytes + y_off[n]);
        for (long long i = threadIdx.x; i < y_len / 4; i += blockDim.x) dst[i] = ys[i];
    }
    if (g.T) {
        // the picture of this tile: header words (first tile), length word t (tile t), and the picture's offset and status
        const int t = n % g.T, n0 = n - t;
        const long long hdr = 4ll * (4 + g.T);
        long long off0, len0;
        image_extent(y_off, z_off, fixed, g.T, n0, &off0, &len0);
        uint32_t* pic = reinterpret_cast<uint32_t*>(out + (off0 - hdr));
        if (threadIdx.x == 0) {
            if (fits) pic[4 + t] = (uint32_t)len;
            if (t == 0 && fits) { pic[0] = kPictureMagic; pic[1] = 1u; pic[2] = g.hw; pic[3] = (uint32_t)g.T; }
            if (n == N - 1) g.offsets[N / g.T] = off + len;
        }
        if (t == 0 && threadIdx.x < 32) {            // one warp: OR of the group's tile status
            int st = 0;
            for (int j = threadIdx.x; j < g.T; j += 32) {
                long long o, l;
                image_extent(y_off, z_off, fixed, g.T, n0 + j, &o, &l);
                st |= y_st[n0 + j] | z_st[n0 + j] | (o + l <= capacity ? 0 : RANS_ST_OVERFLOW);
            }
            st = __reduce_or_sync(0xffffffffu, st);
            if (threadIdx.x == 0) {
                g.offsets[n / g.T] = off0 - hdr;
                g.status[n / g.T] = st;
            }
        }
    }
}

// ranges [4 N]: z begin, z end, y begin, y end of every container (byte offsets into the blob; all 0 for a refused container)
__global__ void __launch_bounds__(256)
image_parse_kernel(const IoBlock* __restrict__ io, ImageFields f, int N, int64_t* __restrict__ ranges) {
    extern __shared__ uint32_t seen[];               // bitmap of the ids met so far, L bits
    __shared__ int s_st;
    const int n = blockIdx.x;
    const int L = f.L, K = f.K, w = f.id_bits, map_words = (L + 31) / 32;
    for (int i = threadIdx.x; i < map_words; i += blockDim.x) seen[i] = 0;
    if (threadIdx.x == 0) s_st = 0;
    const uint8_t* data = io->img_data;
    const long long c0 = io->img_offsets[n], c1 = io->img_ends[n];
    const bool range_ok = c0 >= 0 && c1 >= c0 && c1 <= io->img_n_bytes && !(c0 & 3) && !((c1 - c0) & 3);
    const long long n_words = range_ok ? (c1 - c0) / 4 : 0;
    const uint32_t* cw = reinterpret_cast<const uint32_t*>(data + (range_ok ? c0 : 0));
    int st = 0;
    uint32_t h[kHeaderWords] = {0, 0, 0, 0, 0, 0, 0};
    long long id_words = 0;
    if (n_words < kHeaderWords) {
        st = IMG_ST_HEADER;
    } else {
#pragma unroll
        for (int i = 0; i < kHeaderWords; ++i) h[i] = __ldg(cw + i);
        const long long k_hdr = h[3] & 0xffffu;
        id_words = (k_hdr * w + 31) / 32;
        if (h[0] != kImageMagic || (h[1] & 0xffu) != (f.word1 & 0xffu) || (h[2] >> 24) || (h[3] >> 16) || (h[5] & 3) || (h[6] & 3) ||
            kHeaderWords + id_words + h[5] / 4 + h[6] / 4 != n_words)
            st |= IMG_ST_HEADER;
        if ((h[1] >> 8) != (f.word1 >> 8) || (h[2] & 0xffffffu) != f.word2 || (h[3] & 0xffffu) != f.word3) st |= IMG_ST_CONFIG;
        if (h[4] != f.tag) st |= IMG_ST_MODEL;
    }
    __syncthreads();
    const bool ids_read = !(st & (IMG_ST_HEADER | IMG_ST_CONFIG));     // the section holds K ids of w bits inside the container
    if (ids_read) {
        int bad = 0;
        for (int j = threadIdx.x; j < K; j += blockDim.x) {
            const uint32_t id = unpack_id(cw + kHeaderWords, w, j);
            if (id >= (uint32_t)L) { bad = 1; continue; }
            const uint32_t bit = 1u << (id & 31);
            if (atomicOr(seen + (id >> 5), bit) & bit) bad = 1;
        }
        if (bad) atomicOr(&s_st, IMG_ST_IDS);
    }
    __syncthreads();
    st |= s_st;
    int64_t* restore = io->img_ids_restore + (size_t)n * L;
    int64_t* keep = io->img_ids_keep ? io->img_ids_keep + (size_t)n * K : nullptr;
    if (st == 0) {
        // kept id j at position ids_keep[j]; every other position p, in ascending order, K + (p - kept positions below p)
        for (int p = threadIdx.x; p < L; p += blockDim.x) {
            const uint32_t word = seen[p >> 5], bit = 1u << (p & 31);
            if (word & bit) continue;
            int below = __popc(word & (bit - 1));
            for (int i = 0; i < (p >> 5); ++i) below += __popc(seen[i]);
            restore[p] = K + (p - below);
        }
        for (int j = threadIdx.x; j < K; j += blockDim.x) {
            const uint32_t id = unpack_id(cw + kHeaderWords, w, j);
            restore[id] = j;
            if (keep) keep[j] = id;
        }
    } else {                                          // a refused container: the identity, so that every later read stays in range
        for (int p = threadIdx.x; p < L; p += blockDim.x) restore[p] = p;
        if (keep) for (int j = threadIdx.x; j < K; j += blockDim.x) keep[j] = j;
    }
    if (threadIdx.x == 0) {
        const long long zb = st ? 0 : c0 + 4 * (kHeaderWords + id_words), ze = st ? 0 : zb + h[5], ye = st ? 0 : ze + h[6];
        ranges[n] = zb;
        ranges[N + n] = ze;
        ranges[2 * N + n] = ze;
        ranges[3 * N + n] = ye;
        io->status[n] = st;
    }
}

cudaError_t launch_image_pack(const int64_t* ids_keep, const uint8_t* y_bytes, const int64_t* y_off, const int32_t* y_st,
                              const uint8_t* z_bytes, const int64_t* z_off, const int32_t* z_st, const ImageFields& f, int N,
                              uint8_t* out, long long capacity, int64_t* offsets, int32_t* status, cudaStream_t st,
                              const PictureGroup& g) {
    image_pack_kernel<<<N, 256, 0, st>>>(ids_keep, y_bytes, y_off, y_st, z_bytes, z_off, z_st, f, N, out, capacity, offsets, status, g);
    return cudaGetLastError();
}

cudaError_t launch_image_parse(const IoBlock* io, const ImageFields& f, int N, int64_t* ranges, cudaStream_t st) {
    const size_t smem = (size_t)(f.L + 31) / 32 * 4;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(image_parse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    image_parse_kernel<<<N, 256, smem, st>>>(io, f, N, ranges);
    return cudaGetLastError();
}

}  // namespace tmae
