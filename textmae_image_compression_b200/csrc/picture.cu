// Pictures of any size (DESIGN.md section 7, "The picture container"): tiling.py's policy on the GPU, and the picture container.
// A picture [3, H, W] is zero-padded on the bottom / right and cut into rows x cols tiles of side S = img_size, raster order;
// every tile is coded as one image container.  Little-endian 32-bit words of a picture:
//   0 magic "TMAP" | 1 version (byte 0), reserved (bytes 1-3) | 2 H (16 bits), W (16) | 3 T = rows * cols
//   | 4 .. 4 + T - 1 byte length of every tile container | the T tile containers in raster order
// Tile: cut tiles (and grey tiles) out of the pictures.  Untile: copy the tiles back into the canvas, padding dropped.
// Parse: one CTA per picture, the first stage of the picture decode; it validates the header against the call's geometry and
// hands the container parse the byte range of every tile (empty for a picture it refuses).  Status: after the decode, every
// picture's status ORs in its tiles'.
#include "common.cuh"
#include "kernels.h"

namespace tmae {

namespace {
// cv2.cvtColor(RGB2GRAY) of 8-bit pixels: fixed-point weights 0.299 / 0.587 / 0.114 with 15 fraction bits, rounded
__device__ __forceinline__ uint32_t to_u8(float x) {
    const float v = fminf(fmaxf(rintf(__fmul_rn(x, 255.f)), 0.f), 255.f);      // saturate_cast<uchar>(rint(255 x)); NaN -> 0
    return (uint32_t)v;
}
}  // namespace

// One thread per tile pixel: its three channels, and its grey value (cut from `gray`, or made from the RGB when gray is null).
__global__ void __launch_bounds__(256)
picture_tile_kernel(const float* __restrict__ imgs, const uint8_t* __restrict__ gray, int H, int W, int S, int cols, int T,
                    long long n_pix, float* __restrict__ tiles, uint8_t* __restrict__ gray_tiles) {
    const long long SS = (long long)S * S;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_pix; i += (long long)gridDim.x * blockDim.x) {
        const long long n = i / SS;
        const int yx = (int)(i - n * SS), y = yx / S, x = yx - y * S;
        const long long p = n / T;
        const int t = (int)(n - p * T), Y = (t / cols) * S + y, X = (t % cols) * S + x;
        const bool in = Y < H && X < W;
        const long long hw = (long long)H * W, src = in ? (long long)Y * W + X : 0;
        float v[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c] = in ? imgs[(p * 3 + c) * hw + src] : 0.f;
        if (tiles) {
#pragma unroll
            for (int c = 0; c < 3; ++c) tiles[(n * 3 + c) * SS + yx] = v[c];
        }
        if (gray_tiles) {
            uint32_t g = 0;
            if (in) g = gray ? gray[p * hw + src] : (9798u * to_u8(v[0]) + 19235u * to_u8(v[1]) + 3735u * to_u8(v[2]) + 16384u) >> 15;
            gray_tiles[i] = (uint8_t)g;
        }
    }
}

// One thread per canvas element; 64-bit indexes (P * 3 * H * W may exceed 2^31).
__global__ void __launch_bounds__(256)
picture_untile_kernel(const float* __restrict__ tiles, int H, int W, int S, int cols, int T, long long n_el,
                      float* __restrict__ canvas) {
    const long long hw = (long long)H * W, SS = (long long)S * S;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_el; i += (long long)gridDim.x * blockDim.x) {
        const long long pc = i / hw;                               // picture * 3 + channel
        const long long r = i - pc * hw;
        const int Y = (int)(r / W), X = (int)(r - (long long)Y * W);
        const long long p = pc / 3;
        const int c = (int)(pc - p * 3);
        const long long n = p * T + (Y / S) * cols + X / S;
        canvas[i] = tiles[(n * 3 + c) * SS + (long long)(Y % S) * S + X % S];
    }
}

// io->pic_ranges [2 N]: begin and end byte of every tile container in io->img_data (0, 0 for all tiles of a refused picture);
// io->pic_status[p] = PIC_ST_HEADER or 0.  Grid: one CTA per picture.
__global__ void __launch_bounds__(256)
picture_parse_kernel(const IoBlock* __restrict__ io, int S) {
    __shared__ long long s_part[256];
    __shared__ int s_bad;
    const int p = blockIdx.x;
    const int H = io->pic_H, W = io->pic_W, P = io->pic_P;
    const int cols = (W + S - 1) / S, T = ((H + S - 1) / S) * cols;
    const long long N = (long long)P * T;
    const long long c0 = io->pic_offsets[p], c1 = io->pic_offsets[p + 1];
    const bool range_ok = c0 >= 0 && c1 >= c0 && c1 <= io->img_n_bytes && !(c0 & 3) && !((c1 - c0) & 3);
    const long long n_words = range_ok ? (c1 - c0) / 4 : 0;
    const uint32_t* pw = reinterpret_cast<const uint32_t*>(io->img_data + (range_ok ? c0 : 0));
    const long long hdr = 4ll * (4 + T);
    bool ok = n_words >= 4 + (long long)T;
    if (ok) {
        const uint32_t w0 = __ldg(pw), w1 = __ldg(pw + 1), w2 = __ldg(pw + 2), w3 = __ldg(pw + 3);
        ok = w0 == kPictureMagic && w1 == 1u && (w2 & 0xffffu) == (uint32_t)H && (w2 >> 16) == (uint32_t)W && w3 == (uint32_t)T;
    }
    // every length a multiple of 4, and the lengths add up to the picture: per-thread chunks of the table, then their sums
    const int chunk = (T + blockDim.x - 1) / blockDim.x;
    const int t0 = min(T, (int)threadIdx.x * chunk), t1 = min(T, t0 + chunk);
    long long sum = 0;
    int bad = 0;
    if (ok) {
        for (int t = t0; t < t1; ++t) {
            const uint32_t len = __ldg(pw + 4 + t);
            bad |= len & 3;
            sum += len;
        }
    }
    s_part[threadIdx.x] = sum;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    if (bad) atomicOr(&s_bad, 1);
    long long before = 0, total = 0;                 // exclusive prefix of this thread's chunk, and the whole table's sum
    for (int i = 0; i < (int)blockDim.x; ++i) {
        if (i < (int)threadIdx.x) before += s_part[i];
        total += s_part[i];
    }
    __syncthreads();
    ok = ok && !s_bad && hdr + total == c1 - c0;
    int64_t* begins = io->pic_ranges;
    int64_t* ends = io->pic_ranges + N;
    long long b = c0 + hdr + before;
    for (int t = t0; t < t1; ++t) {
        const long long n = (long long)p * T + t;
        const long long len = ok ? (long long)__ldg(pw + 4 + t) : 0;
        begins[n] = ok ? b : 0;
        ends[n] = ok ? b + len : 0;
        b += len;
    }
    if (threadIdx.x == 0) io->pic_status[p] = ok ? 0 : PIC_ST_HEADER;
}

// io->pic_status[p] |= the status of each of its T tiles (io->status).  Grid: one CTA per picture.
__global__ void __launch_bounds__(256)
picture_status_kernel(const IoBlock* __restrict__ io, int T) {
    __shared__ int s_st;
    if (threadIdx.x == 0) s_st = 0;
    __syncthreads();
    const long long n0 = (long long)blockIdx.x * T;
    int st = 0;
    for (int t = threadIdx.x; t < T; t += blockDim.x) st |= io->status[n0 + t];
    if (st) atomicOr(&s_st, st);
    __syncthreads();
    if (threadIdx.x == 0) io->pic_status[blockIdx.x] |= s_st;
}

namespace {
int grid_for(long long n) {
    const long long b = (n + 255) / 256;
    return (int)(b < 1 ? 1 : b > 148 * 64 ? 148 * 64 : b);
}
}  // namespace

cudaError_t launch_picture_tile(const float* imgs, const uint8_t* gray, int P, int H, int W, int S, float* tiles,
                                uint8_t* gray_tiles, cudaStream_t st) {
    const int cols = (W + S - 1) / S, T = ((H + S - 1) / S) * cols;
    const long long n_pix = (long long)P * T * S * S;
    picture_tile_kernel<<<grid_for(n_pix), 256, 0, st>>>(imgs, gray, H, W, S, cols, T, n_pix, tiles, gray_tiles);
    return cudaGetLastError();
}

cudaError_t launch_picture_untile(const float* tiles, int P, int H, int W, int S, float* canvas, cudaStream_t st) {
    const int cols = (W + S - 1) / S, T = ((H + S - 1) / S) * cols;
    const long long n_el = (long long)P * 3 * H * W;
    picture_untile_kernel<<<grid_for(n_el), 256, 0, st>>>(tiles, H, W, S, cols, T, n_el, canvas);
    return cudaGetLastError();
}

cudaError_t launch_picture_parse(const IoBlock* io, int P, int S, cudaStream_t st) {
    picture_parse_kernel<<<P, 256, 0, st>>>(io, S);
    return cudaGetLastError();
}

cudaError_t launch_picture_status(const IoBlock* io, int P, int T, cudaStream_t st) {
    picture_status_kernel<<<P, 256, 0, st>>>(io, T);
    return cudaGetLastError();
}

}  // namespace tmae
