// gb_frames.cu -- batched frame capture (gbenv_capture_frames) and decode (gbenv_frames_to_rgb), linked into libgbenv.so
// next to gbenv.cu.
//
// A packed frame is an env's framebuffer as the emulator keeps it (gb_layout.cuh): 144 lines x FB_LINE_WORDS words, the
// pixel (x, y) is the 2-bit shade at bit 2 * (x & 15) of word y * FB_LINE_WORDS + x / 16.  In the device arrays word w of
// env e sits at il_index(e / 32, FB_WORDS, w, e % 32); a captured frame is the same FB_WORDS words made contiguous.
#include <stdint.h>
#include "../../include/gbenv.h"
#include "gb_frames.cuh"
#include "gb_layout.cuh"

#define FRAMES_TILE 32      // list entries x words per block of k_frames_capture
#define FRAMES_ROWS 8       // threadIdx.y extent: each thread moves FRAMES_TILE / FRAMES_ROWS words
#define FRAMES_RGB_THREADS 256
static_assert(FB_WORDS == GBENV_FRAME_WORDS, "a packed frame is the framebuffer as stored");
static_assert(FB_WORDS % FRAMES_TILE == 0, "a block's words never straddle the end of a frame");

// grid: (ceil(n / 32), FB_WORDS / 32), block (32, 8).  Reads: lane x takes word w of list entry x, so the 32 lanes of a warp
// read one 128-byte line when the entries are the 32 envs of one tile, in order.  Writes: after a transpose through shared
// memory, lane x writes word x of one entry, so every warp store is one 128-byte line whatever the ids.  Entries whose id is
// outside [0, n_envs) are neither read nor written.
__global__ void __launch_bounds__(FRAMES_TILE * FRAMES_ROWS) k_frames_capture(const uint32_t *__restrict__ fb, const int32_t *__restrict__ ids, int n,
                                                                             int n_envs, uint32_t *__restrict__ frames) {
    __shared__ uint32_t s_words[FRAMES_TILE][FRAMES_TILE + 1];  // [word][entry], padded against bank conflicts
    __shared__ int s_env[FRAMES_TILE];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int first = blockIdx.x * FRAMES_TILE;
    const uint32_t w0 = blockIdx.y * FRAMES_TILE;
    if (ty == 0) {
        const int i = first + tx;
        int env = -1;
        if (i < n) env = ids ? ids[i] : i;
        s_env[tx] = env >= 0 && env < n_envs ? env : -1;
    }
    __syncthreads();
    const int env = s_env[tx];
    if (env >= 0) {
        const uint32_t *src = fb + il_index(env >> 5, FB_WORDS, w0, env & 31);
#pragma unroll
        for (int k = ty; k < FRAMES_TILE; k += FRAMES_ROWS) s_words[k][tx] = src[(size_t)k * GB_TILE];
    }
    __syncthreads();
#pragma unroll
    for (int k = ty; k < FRAMES_TILE; k += FRAMES_ROWS)
        if (s_env[k] >= 0) frames[(size_t)(first + k) * FB_WORDS + w0 + tx] = s_words[tx][k];
}

// One thread per packed word, i.e. 16 consecutive pixels of one line.  Pixel (x, y) of frame f is pixel number
// 16 * (f * FB_WORDS + y * FB_LINE_WORDS + x / 16) + x % 16 of the output, so word g expands to the bytes
// [16 * g * channels, 16 * (g + 1) * channels): one 16-byte store for grey, three for RGB.  `out` is 16-byte aligned.
__global__ void __launch_bounds__(FRAMES_RGB_THREADS) k_frames_to_rgb(const uint32_t *__restrict__ frames, size_t n_words, int channels,
                                                                      uint8_t *__restrict__ out) {
    const size_t g = (size_t)blockIdx.x * FRAMES_RGB_THREADS + threadIdx.x;
    if (g >= n_words) return;
    const uint32_t v = frames[g];
    const uint32_t GREY = 0x005599FFu;  // byte s = the grey of shade s: {0xFF, 0x99, 0x55, 0x00}, as gbenv_screen
    uint32_t q[4];  // the 16 grey bytes, little-endian
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint32_t b = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) b |= ((GREY >> (8 * ((v >> (2 * (4 * k + j))) & 3))) & 0xFF) << (8 * j);
        q[k] = b;
    }
    if (channels == 1) {
        reinterpret_cast<uint4 *>(out)[g] = make_uint4(q[0], q[1], q[2], q[3]);
        return;
    }
    // RGB: every grey byte three times.  Output byte 3 * p + c is grey byte p; word m of the 12 holds bytes 4m .. 4m + 3.
    uint32_t r[12];
#pragma unroll
    for (int m = 0; m < 12; m++) {
        uint32_t b = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int p = (4 * m + j) / 3;
            b |= ((q[p >> 2] >> (8 * (p & 3))) & 0xFF) << (8 * j);
        }
        r[m] = b;
    }
    uint4 *dst = reinterpret_cast<uint4 *>(out) + 3 * g;
    dst[0] = make_uint4(r[0], r[1], r[2], r[3]);
    dst[1] = make_uint4(r[4], r[5], r[6], r[7]);
    dst[2] = make_uint4(r[8], r[9], r[10], r[11]);
}

cudaError_t launch_frames_capture(const uint32_t *fb, const int32_t *ids, int n, int n_envs, uint32_t *frames, cudaStream_t st) {
    const dim3 grid((n + FRAMES_TILE - 1) / FRAMES_TILE, FB_WORDS / FRAMES_TILE), block(FRAMES_TILE, FRAMES_ROWS);
    k_frames_capture<<<grid, block, 0, st>>>(fb, ids, n, n_envs, frames);
    return cudaGetLastError();
}

cudaError_t launch_frames_to_rgb(const uint32_t *frames, int n_frames, int channels, uint8_t *out, cudaStream_t st) {
    const size_t words = (size_t)n_frames * FB_WORDS;
    k_frames_to_rgb<<<(unsigned)((words + FRAMES_RGB_THREADS - 1) / FRAMES_RGB_THREADS), FRAMES_RGB_THREADS, 0, st>>>(frames, words, channels, out);
    return cudaGetLastError();
}
