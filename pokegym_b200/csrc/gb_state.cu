// gb_state.cu -- the PyBoy v9 file of a list of envs (gbenv_save_states), linked into libgbenv.so next to gbenv.cu.
//
// The file layout is STATE_LAYOUT (gb_image.h), the same table image_to_blob serialises from.  Output row i is the file of
// list entry i, rows back to back, so row i starts at byte i * GBENV_STATE_BYTES = 2i (mod 16) of the 16-byte aligned output,
// and the sections of a row start at unaligned offsets too.  The kernel therefore writes the flat output in aligned 16-byte
// units and derives each byte's (row, file offset), and from that its source, from the unit's address.
#include <stdint.h>
#include "../../include/gbenv.h"
#include "gb_image.h"
#include "gb_state.cuh"

#define SAVE_CHUNK 1024  // file bytes per block (per list entry)
#define SAVE_CHUNKS ((GBENV_STATE_BYTES + SAVE_CHUNK - 1) / SAVE_CHUNK)
#define SAVE_WARPS 8
#define SAVE_MAX_WINDOWS 256

// Which image words a block stages in shared memory.  Block (x, k) handles file bytes [k * SAVE_CHUNK, +SAVE_CHUNK) of 32 list
// entries.  For each section that overlaps the chunk, one window: the image words of the section's bytes from the chunk start
// to 15 bytes past the chunk end (a 16-byte unit that starts in the chunk and stays in the section is then fully staged).
struct SavePlan {
    uint16_t sec0[SAVE_CHUNKS], nsec[SAVE_CHUNKS], win0[SAVE_CHUNKS];  // sections sec0 .. sec0 + nsec - 1 <-> windows win0 ..
    uint32_t jlo[SAVE_MAX_WINDOWS], n[SAVE_MAX_WINDOWS], base[SAVE_MAX_WINDOWS];  // image words jlo .. jlo + n - 1 at smem word base
    uint32_t n_windows, max_words;
};

constexpr SavePlan make_save_plan() {
    SavePlan p{};
    uint32_t w = 0;
    for (uint32_t k = 0; k < SAVE_CHUNKS; k++) {
        const uint32_t o0 = k * SAVE_CHUNK, o1 = o0 + SAVE_CHUNK < GBENV_STATE_BYTES ? o0 + SAVE_CHUNK : GBENV_STATE_BYTES;
        const int sec0 = state_section_of(STATE_LAYOUT, o0);
        p.sec0[k] = (uint16_t)sec0;
        p.win0[k] = (uint16_t)w;
        uint32_t words = 0;
        int i = sec0;
        for (; i < STATE_SECTIONS && STATE_LAYOUT.s[i].off < o1; i++, w++) {
            const StateSection &s = STATE_LAYOUT.s[i];
            const uint32_t lo = o0 > s.off ? o0 : s.off, end = s.off + s.len, hi = (o1 + 15 < end ? o1 + 15 : end) - 1;
            p.base[w] = words;
            p.jlo[w] = s.kind == SK_CONST ? 0 : state_word(s, lo);
            p.n[w] = s.kind == SK_CONST ? 0 : state_word(s, hi) - p.jlo[w] + 1;
            words += p.n[w];
        }
        p.nsec[k] = (uint16_t)(i - sec0);
        if (words > p.max_words) p.max_words = words;
    }
    p.n_windows = w;
    return p;
}

static constexpr SavePlan SAVE_PLAN = make_save_plan();
static_assert(SAVE_PLAN.n_windows <= SAVE_MAX_WINDOWS, "raise SAVE_MAX_WINDOWS");
// an entry's staged words, with room for the one word past a window that the unit loops read (and ignore) at shift 0; odd,
// so the 32 entries of a staging store fall in 32 different banks
#define SAVE_ROW ((SAVE_PLAN.max_words + 2) | 1)
static_assert(GB_TILE * SAVE_ROW * 4 <= 48 * 1024, "staging fits the static shared-memory limit");

static __constant__ StateLayout c_layout = STATE_LAYOUT;
static __constant__ SavePlan c_plan = SAVE_PLAN;

__device__ __forceinline__ int save_env(const int32_t *ids, int id0, int i, int n_envs) {
    const int env = ids ? ids[i] : id0 + i;
    return env >= 0 && env < n_envs ? env : -1;
}

// A unit the fast path does not take: it spans sections or rows, or lies in a section of single fields or scanline records.
// Each byte finds its own row and section; bytes of this entry in a staged window come from shared memory, the others (the
// next row's first bytes, a section that starts past the chunk) from the interleaved arrays.  Bytes of a row with an id
// outside [0, n_envs), or past the last row, are not written.
static __device__ __noinline__ void save_unit_slow(const DevArrays d, const int32_t *__restrict__ ids, int id0, int n, int k_chunk, int row,
                                                   int env, const uint32_t *srow, uint32_t o, uint8_t *__restrict__ dst) {
    uint32_t q[4] = {0, 0, 0, 0}, valid = 0;
    int next_env = -2;
    const uint32_t sec0 = c_plan.sec0[k_chunk], nsec = c_plan.nsec[k_chunk], win0 = c_plan.win0[k_chunk];
    const uint32_t staged_end = (uint32_t)k_chunk * SAVE_CHUNK + SAVE_CHUNK + 15;
#pragma unroll
    for (int b = 0; b < 16; b++) {
        uint32_t ob = o + b;
        int e = env;
        bool own = true;
        if (ob >= GBENV_STATE_BYTES) {
            if (row + 1 >= n) break;  // the output ends with the last row
            if (next_env == -2) next_env = save_env(ids, id0, row + 1, d.n_envs);
            ob -= GBENV_STATE_BYTES;
            e = next_env;
            own = false;
        }
        if (e < 0) continue;
        const int si = state_section_of(c_layout, ob);
        const StateSection s = c_layout.s[si];
        uint32_t w = 0;
        if (s.kind != SK_CONST) {
            const uint32_t j = state_word(s, ob), m = (uint32_t)si - sec0;
            if (own && m < nsec && ob < staged_end) w = srow[c_plan.base[win0 + m] + j - c_plan.jlo[win0 + m]];
            else w = __ldg(image_slot(d, e, j));
        }
        q[b >> 2] |= (uint32_t)state_byte(s, ob, w) << (8 * (b & 3));
        valid |= 1u << b;
    }
    if (valid == 0xFFFFu) {
        *reinterpret_cast<uint4 *>(dst) = make_uint4(q[0], q[1], q[2], q[3]);
        return;
    }
#pragma unroll
    for (int b = 0; b < 16; b++)
        if ((valid >> b) & 1) dst[b] = (uint8_t)(q[b >> 2] >> (8 * (b & 3)));
}

// grid (ceil(n / 32), SAVE_CHUNKS), block (32, SAVE_WARPS).
// Staging: lane x loads the window words of list entry x, so when the entries are the 32 envs of one tile in order every warp
// load is one 128-byte line; the words go to shared memory, one row per entry.
// Writing: warp y takes entries y, y + 8, ..; its lanes take consecutive 16-byte units of the entry's row, so every warp store
// covers 512 contiguous bytes.  A unit belongs to the block holding its first byte.  Inside one section of RAM bytes (VRAM,
// WRAM, cartridge RAM, ...) or of the screen -- all but ~100 of a row's 8,914 units -- it is assembled from staged words with
// funnel shifts; the rest go through save_unit_slow.
__global__ void __launch_bounds__(GB_TILE * SAVE_WARPS) k_save_states(const DevArrays d, const int32_t *__restrict__ ids, int id0, int n,
                                                                     uint8_t *__restrict__ blobs) {
    __shared__ uint32_t s_img[GB_TILE * SAVE_ROW];
    __shared__ int s_env[GB_TILE];
    const int tx = threadIdx.x, ty = threadIdx.y, first = blockIdx.x * GB_TILE, k_chunk = blockIdx.y;
    const uint32_t sec0 = c_plan.sec0[k_chunk], nsec = c_plan.nsec[k_chunk], win0 = c_plan.win0[k_chunk];
    if (ty == 0) s_env[tx] = first + tx < n ? save_env(ids, id0, first + tx, d.n_envs) : -1;
    __syncthreads();
    {
        const int env = s_env[tx];
        if (env >= 0) {
            for (uint32_t m = 0; m < nsec; m++) {
                const uint32_t jlo = c_plan.jlo[win0 + m], cnt = c_plan.n[win0 + m], base = c_plan.base[win0 + m];
                for (uint32_t i = ty; i < cnt; i += SAVE_WARPS) s_img[tx * SAVE_ROW + base + i] = __ldg(image_slot(d, env, jlo + i));
            }
        }
    }
    __syncthreads();
    const uint32_t o0 = (uint32_t)k_chunk * SAVE_CHUNK, o1 = o0 + SAVE_CHUNK < GBENV_STATE_BYTES ? o0 + SAVE_CHUNK : GBENV_STATE_BYTES;
    for (int k = ty; k < GB_TILE && first + k < n; k += SAVE_WARPS) {
        const int row = first + k, env = s_env[k];
        const size_t row0 = (size_t)row * GBENV_STATE_BYTES;
        const size_t u0 = (row0 + o0 + 15) >> 4, u1 = (row0 + o1 + 15) >> 4;
        const uint32_t *srow = s_img + k * SAVE_ROW;
        for (size_t u = u0 + tx; u < u1; u += 32) {
            const uint32_t o = (uint32_t)((u << 4) - row0);
            uint8_t *dst = blobs + (u << 4);
            if (env < 0) {
                if (o + 16 > GBENV_STATE_BYTES) save_unit_slow(d, ids, id0, n, k_chunk, row, env, srow, o, dst);  // the next row's head
                continue;
            }
            uint32_t m = 0;
            while (m + 1 < nsec && c_layout.s[sec0 + m + 1].off <= o) m++;
            const StateSection s = c_layout.s[sec0 + m];
            const uint32_t r = o - s.off, jlo = c_plan.jlo[win0 + m], base = c_plan.base[win0 + m];
            if (r + 16 > s.len || (s.kind != SK_BYTES && s.kind != SK_FB)) {
                save_unit_slow(d, ids, id0, n, k_chunk, row, env, srow, o, dst);
                continue;
            }
            uint32_t v[5];
            uint32_t sh;
            if (s.kind == SK_BYTES) {
                const uint32_t a = s.src + r, wi = base + (a >> 2) - jlo;
                sh = 8 * (a & 3);
#pragma unroll
                for (int t = 0; t < 5; t++) v[t] = srow[wi + t];
            } else {
                const uint32_t p0 = r >> 2;
                sh = 8 * (r & 3);
#pragma unroll
                for (int t = 0; t < 5; t++) {
                    const uint32_t p = p0 + t, word = srow[base + IMG_FB + (p >> 4) - jlo];
                    v[t] = state_shade_word((word >> (2 * (p & 15))) & 3);
                }
            }
            *reinterpret_cast<uint4 *>(dst) = make_uint4(__funnelshift_r(v[0], v[1], sh), __funnelshift_r(v[1], v[2], sh),
                                                         __funnelshift_r(v[2], v[3], sh), __funnelshift_r(v[3], v[4], sh));
        }
    }
}

cudaError_t launch_save_states(const DevArrays &d, const int32_t *ids, int id0, int n, uint8_t *blobs, cudaStream_t st) {
    k_save_states<<<dim3((n + GB_TILE - 1) / GB_TILE, SAVE_CHUNKS), dim3(GB_TILE, SAVE_WARPS), 0, st>>>(d, ids, id0, n, blobs);
    return cudaGetLastError();
}
