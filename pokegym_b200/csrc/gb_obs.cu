// gb_obs.cu -- packed observations (gbenv_step_packed / gbenv_reset_packed / gbenv_unpack_obs), linked into libgbenv.so next
// to gbenv.cu.
//
// The reference observation (k_wrap_obs, gb_wrap.cuh) is uint8 [72][80][4]: channels 0-2 the grey of framebuffer pixel
// (2j, 2i), one of four levels, channel 3 the visited bit of map cell (r - 36 + i, c - 40 + j) as 0 / 255.  So 3 bits per
// pixel carry all of it.  A packed row i is 8 words: words 0-4 the 80 shades at 2 bits each (the framebuffer's own
// encoding), words 5-7 the 80 visited bits; 2,304 B per env instead of 23,040 (include/gbenv.h has the exact layout).
#include <stdint.h>
#include "../../include/gbenv.h"
#include "gb_layout.cuh"
#include "gb_obs.cuh"

#define OBS_PACK_ROWS 8       // threadIdx.y extent of k_obs_pack: obs rows per block
#define OBS_ROW_WORDS 8       // packed words per obs row
#define OBS_SHADE_WORDS 5     // of which shades
#define OBS_CHUNKS_PER_ROW 20 // 16-byte chunks (4 pixels) of a reference obs row
#define OBS_UNPACK_THREADS 256
static_assert(GBENV_OBS_PACKED_WORDS == GBENV_OBS_H * OBS_ROW_WORDS && GBENV_OBS_PACKED_BYTES == 4 * GBENV_OBS_PACKED_WORDS, "packed row layout");
static_assert(GBENV_OBS_H % OBS_PACK_ROWS == 0, "a block's rows never run past the last obs row");
static_assert(GBENV_OBS_W * GBENV_OBS_C == 16 * OBS_CHUNKS_PER_ROW, "a reference obs row is whole 16-byte chunks");
static_assert(2 * GBENV_OBS_W == 16 * FB_LINE_WORDS && GBENV_OBS_W == 16 * OBS_SHADE_WORDS, "two framebuffer words give one word of shades");

// 2-bit fields 0, 2, 4, ..., 14 of v (the even pixels of a framebuffer word) -> fields 0 .. 7 of the result
__device__ __forceinline__ uint32_t even_fields(uint32_t v) {
    v &= 0x33333333u;
    v = (v | (v >> 2)) & 0x0F0F0F0Fu;
    v = (v | (v >> 4)) & 0x00FF00FFu;
    return (v | (v >> 8)) & 0x0000FFFFu;
}

// One thread per (env, obs row): grid (n_tiles, 72 / OBS_PACK_ROWS), block (32, OBS_PACK_ROWS), lane = env within its tile,
// so every load of `mem` and `fb` by a warp is one whole 128-byte line.  Edge rules are k_wrap_obs's: position from D361 /
// D362 / D35E with the map clamped to 247; bitmap rows and columns outside [0, 255), and missing pages, read as 0.
__global__ void __launch_bounds__(32 * OBS_PACK_ROWS) k_obs_pack(const uint32_t *__restrict__ mem, const uint32_t *__restrict__ fb,
                                                                 const uint32_t *__restrict__ vis_pt, const uint32_t *__restrict__ vis_pool, int n_envs,
                                                                 const uint8_t *__restrict__ mask, int invert, uint32_t *__restrict__ packed) {
    const int tile = blockIdx.x, lane = threadIdx.x, env = tile * GB_TILE + lane;
    const int i = blockIdx.y * OBS_PACK_ROWS + threadIdx.y;
    if (env >= n_envs || (mask && (mask[env] != 0) == (invert != 0))) return;
    const uint8_t *memb = (const uint8_t *)(mem + il_index(tile, MEM_WORDS, 0, lane));
    auto rd = [&](uint32_t a) { const uint32_t k = MEM_WRAM + (a - 0xC000u); return (int)memb[((k >> 2) << 7) | (k & 3)]; };
    const int r = rd(0xD361), c = rd(0xD362), map_n = min(rd(0xD35E), WRAP_MAPS - 1);

    uint32_t fw[FB_LINE_WORDS];  // framebuffer line 2i
#pragma unroll
    for (int w = 0; w < FB_LINE_WORDS; w++) fw[w] = fb[il_index(tile, FB_WORDS, (uint32_t)(2 * i) * FB_LINE_WORDS + w, lane)];

    // visited window: columns c-40 .. c+39 of bitmap row r-36+i
    uint32_t win0 = 0, win1 = 0, win2 = 0;
    const int rr = r - 36 + i;
    const uint32_t pg = (rr >= 0 && rr < 255) ? vis_pt[(size_t)env * VIS_PT_ENTRIES + map_n * VIS_BANDS + rr / VIS_BAND_ROWS] : 0u;
    if (pg) {
        const uint4 *row = (const uint4 *)(vis_pool + (size_t)(pg - 1) * VIS_PAGE_WORDS + (rr % VIS_BAND_ROWS) * VIS_ROW_WORDS);
        const uint4 a = row[0], b = row[1];
        // the row with two zero words on either side (column x is bit x + 64); column 255 reads as 0
        const uint32_t e[12] = {0u, 0u, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w & 0x7FFFFFFFu, 0u, 0u};
        const int s = c - 40 + 64, q = s >> 5;  // the window starts at bit s of e[]: s in 24 .. 279, q in 0 .. 8
        const uint32_t sh = (uint32_t)s & 31u;
        uint32_t x0 = 0, x1 = 0, x2 = 0, x3 = 0;  // e[q .. q+3], by selection: an indexed register array would go to local memory
#pragma unroll
        for (int k = 0; k <= 8; k++)
            if (q == k) { x0 = e[k]; x1 = e[k + 1]; x2 = e[k + 2]; x3 = e[k + 3]; }
        win0 = __funnelshift_r(x0, x1, sh);
        win1 = __funnelshift_r(x1, x2, sh);
        win2 = __funnelshift_r(x2, x3, sh) & 0xFFFFu;  // pixels 80 .. 95 do not exist
    }
    uint4 *dst = (uint4 *)(packed + (size_t)env * GBENV_OBS_PACKED_WORDS + i * OBS_ROW_WORDS);
    dst[0] = make_uint4(even_fields(fw[0]) | even_fields(fw[1]) << 16, even_fields(fw[2]) | even_fields(fw[3]) << 16,
                        even_fields(fw[4]) | even_fields(fw[5]) << 16, even_fields(fw[6]) | even_fields(fw[7]) << 16);
    dst[1] = make_uint4(even_fields(fw[8]) | even_fields(fw[9]) << 16, win0, win1, win2);
}

// One thread per 16-byte chunk of the reference output, i.e. 4 pixels of one row: chunk g of the output is bytes
// [16 g, 16 g + 16), pixels j0 .. j0 + 3 of row i of env g / 1440 with i = (g % 1440) / 20, j0 = 4 * (g % 20).
__global__ void __launch_bounds__(OBS_UNPACK_THREADS) k_obs_unpack(const uint32_t *__restrict__ packed, size_t n_chunks, uint8_t *__restrict__ out) {
    const size_t g = (size_t)blockIdx.x * OBS_UNPACK_THREADS + threadIdx.x;
    if (g >= n_chunks) return;
    const size_t row = g / OBS_CHUNKS_PER_ROW;  // env * 72 + i
    const uint32_t j0 = 4 * (uint32_t)(g - row * OBS_CHUNKS_PER_ROW);
    const uint32_t *src = packed + row * OBS_ROW_WORDS;
    const uint32_t shades = __ldg(src + (j0 >> 4)) >> (2 * (j0 & 15));
    const uint32_t vis = __ldg(src + OBS_SHADE_WORDS + (j0 >> 5)) >> (j0 & 31);
    const uint32_t GREY = 0x005599FFu;  // byte s = the grey of shade s: {0xFF, 0x99, 0x55, 0x00}
    uint32_t px[4];
#pragma unroll
    for (int t = 0; t < 4; t++)
        px[t] = ((GREY >> (8 * ((shades >> (2 * t)) & 3))) & 0xFFu) * 0x010101u | (((vis >> t) & 1u) ? 0xFF000000u : 0u);
    reinterpret_cast<uint4 *>(out)[g] = make_uint4(px[0], px[1], px[2], px[3]);
}

cudaError_t launch_obs_pack(const uint32_t *mem, const uint32_t *fb, const uint32_t *vis_pt, const uint32_t *vis_pool, int n_envs, int n_tiles,
                            const uint8_t *mask, int invert, uint32_t *packed, cudaStream_t st) {
    const dim3 grid(n_tiles, GBENV_OBS_H / OBS_PACK_ROWS), block(GB_TILE, OBS_PACK_ROWS);
    k_obs_pack<<<grid, block, 0, st>>>(mem, fb, vis_pt, vis_pool, n_envs, mask, invert, packed);
    return cudaGetLastError();
}

cudaError_t launch_obs_unpack(const uint32_t *packed, int n, uint8_t *out, cudaStream_t st) {
    const size_t chunks = (size_t)n * GBENV_OBS_H * OBS_CHUNKS_PER_ROW;
    k_obs_unpack<<<(unsigned)((chunks + OBS_UNPACK_THREADS - 1) / OBS_UNPACK_THREADS), OBS_UNPACK_THREADS, 0, st>>>(packed, chunks, out);
    return cudaGetLastError();
}
