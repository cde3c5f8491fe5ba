// gb_state.cu -- the PyBoy v9 file of a list of envs (gbenv_save_states) and back (gbenv_load_states), linked into
// libgbenv.so next to gbenv.cu.
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

// ---------------------------------------------------------------------------------------------------- gbenv_load_states
// The reverse direction: rows (v9 files, laid out as k_save_states writes them) into the envs' state.  k_load_check decides
// which entry each env takes, before anything is written; k_load_states then writes the image words of those entries.

#define LOAD_CHUNK 1024  // file bytes of a bulk section per block (per list entry)
#define LOAD_WARPS 8
#define LOAD_CHECK_WARPS 8
#define LOAD_MAX_CHUNKS 160
#define LOAD_MAX_SEGS 160
#define LOAD_MAX_WINS 160

// Which image words a block writes and which file bytes it stages for them.  The bulk sections (RAM runs of at least
// LOAD_CHUNK bytes, and the screen) are cut into LOAD_CHUNK-byte pieces, one chunk each: one window of file bytes, one
// segment of whole image words.  The last chunk takes every other image word, in segments split at the image regions,
// each with the sections that can feed it, and stages the file runs of all other sections.
struct LoadPlan {
    uint16_t seg0[LOAD_MAX_CHUNKS], nseg[LOAD_MAX_CHUNKS], win0[LOAD_MAX_CHUNKS], nwin[LOAD_MAX_CHUNKS];
    uint32_t j0[LOAD_MAX_SEGS], j1[LOAD_MAX_SEGS];  // segment: image words j0 .. j1 - 1, fed by the sections in secs
    uint64_t secs[LOAD_MAX_SEGS];
    uint32_t lo[LOAD_MAX_WINS], hi[LOAD_MAX_WINS], base[LOAD_MAX_WINS];  // window: file bytes [lo, hi), staged at smem word base
    uint32_t n_chunks, max_words;
};

constexpr bool load_bulk(const StateSection &s) {
    return (s.kind == SK_BYTES && s.len >= LOAD_CHUNK) || s.kind == SK_FB;
}
// image words [w0, w1] a section gives bits to (w0 > w1: none)
constexpr void load_image_range(const StateSection &s, uint32_t &w0, uint32_t &w1) {
    w0 = 1;
    w1 = 0;
    if (s.kind == SK_BYTES) { w0 = s.src >> 2; w1 = (s.src + s.len - 1) >> 2; }
    if (s.kind == SK_FIELD) { w0 = w1 = s.src; }
    if (s.kind == SK_LP) { w0 = IMG_LP; w1 = IMG_LP + LP_WORDS - 1; }
    if (s.kind == SK_FB) { w0 = IMG_FB; w1 = IMG_FB + FB_WORDS - 1; }
}
// staged words of a window: the aligned 16-byte units over [lo, hi + 3) at any row alignment
constexpr uint32_t load_window_words(uint32_t lo, uint32_t hi) { return 4 * ((hi - lo + 3 + 15 + 15) / 16); }

constexpr LoadPlan make_load_plan() {
    LoadPlan p{};
    uint32_t c = 0, sg = 0, wn = 0;
    for (int i = 0; i < STATE_SECTIONS; i++) {
        const StateSection &s = STATE_LAYOUT.s[i];
        if (!load_bulk(s)) continue;
        const uint32_t bytes_per_word = s.kind == SK_FB ? 64 : 4;
        for (uint32_t o = 0; o < s.len; o += LOAD_CHUNK, c++, sg++, wn++) {
            const uint32_t e = o + LOAD_CHUNK < s.len ? o + LOAD_CHUNK : s.len;
            const uint32_t w0 = s.kind == SK_FB ? IMG_FB : s.src >> 2;
            p.seg0[c] = (uint16_t)sg; p.nseg[c] = 1; p.win0[c] = (uint16_t)wn; p.nwin[c] = 1;
            p.j0[sg] = w0 + o / bytes_per_word; p.j1[sg] = w0 + e / bytes_per_word; p.secs[sg] = 1ull << i;
            p.lo[wn] = s.off + o; p.hi[wn] = s.off + e; p.base[wn] = 0;
            if (load_window_words(s.off + o, s.off + e) > p.max_words) p.max_words = load_window_words(s.off + o, s.off + e);
        }
    }
    // the last chunk: image words outside the bulk sections, in segments that do not cross a region boundary
    uint32_t cut[32] = {0, IMG_CRAM, IMG_FB, IMG_LP, IMG_REGS, IMG_WORDS};
    uint32_t ncut = 6;
    for (int i = 0; i < STATE_SECTIONS; i++) {
        uint32_t w0 = 0, w1 = 0;
        load_image_range(STATE_LAYOUT.s[i], w0, w1);
        if (load_bulk(STATE_LAYOUT.s[i])) { cut[ncut++] = w0; cut[ncut++] = w1 + 1; }
    }
    for (uint32_t a = 1; a < ncut; a++)  // sort
        for (uint32_t b = a; b > 0 && cut[b - 1] > cut[b]; b--) { const uint32_t t = cut[b]; cut[b] = cut[b - 1]; cut[b - 1] = t; }
    p.seg0[c] = (uint16_t)sg;
    p.win0[c] = (uint16_t)wn;
    for (uint32_t a = 0; a + 1 < ncut; a++) {
        const uint32_t lo = cut[a], hi = cut[a + 1];
        bool bulk = false;
        uint64_t secs = 0;
        for (int i = 0; i < STATE_SECTIONS; i++) {
            uint32_t w0 = 0, w1 = 0;
            load_image_range(STATE_LAYOUT.s[i], w0, w1);
            if (w0 > w1 || w1 < lo || w0 >= hi) continue;
            if (load_bulk(STATE_LAYOUT.s[i])) bulk = true;
            else secs |= 1ull << i;
        }
        if (lo == hi || bulk) continue;
        p.j0[sg] = lo; p.j1[sg] = hi; p.secs[sg] = secs;
        sg++;
    }
    p.nseg[c] = (uint16_t)(sg - p.seg0[c]);
    uint32_t words = 0;
    for (int i = 0; i < STATE_SECTIONS; i++) {  // windows: the file runs of the other sections, adjacent ones merged
        const StateSection &s = STATE_LAYOUT.s[i];
        if (load_bulk(s)) continue;
        if (wn > p.win0[c] && p.hi[wn - 1] == s.off) { p.hi[wn - 1] = s.off + s.len; continue; }
        p.lo[wn] = s.off; p.hi[wn] = s.off + s.len;
        wn++;
    }
    p.nwin[c] = (uint16_t)(wn - p.win0[c]);
    for (uint32_t m = p.win0[c]; m < wn; m++) { p.base[m] = words; words += load_window_words(p.lo[m], p.hi[m]); }
    if (words > p.max_words) p.max_words = words;
    p.n_chunks = c + 1;
    return p;
}

static constexpr LoadPlan LOAD_PLAN = make_load_plan();
static_assert(LOAD_PLAN.n_chunks <= LOAD_MAX_CHUNKS && LOAD_PLAN.seg0[LOAD_PLAN.n_chunks - 1] + LOAD_PLAN.nseg[LOAD_PLAN.n_chunks - 1] <= LOAD_MAX_SEGS &&
              LOAD_PLAN.win0[LOAD_PLAN.n_chunks - 1] + LOAD_PLAN.nwin[LOAD_PLAN.n_chunks - 1] <= LOAD_MAX_WINS, "raise the LOAD_MAX_* limits");
// odd, so that the lanes of a warp, one entry each, read different banks; at least one word past the last window, which a
// file word that starts on a word boundary reads (and ignores)
#define LOAD_ROW ((LOAD_PLAN.max_words + 1) | 1)
static_assert(GB_TILE * LOAD_ROW * 4 <= 48 * 1024, "staging fits the static shared-memory limit");

static __constant__ LoadPlan c_lplan = LOAD_PLAN;

__host__ __device__ constexpr unsigned long long load_key(uint32_t seq, int i) { return ((unsigned long long)seq << 32) | (uint32_t)i; }

// grid ceil(n / LOAD_CHECK_WARPS), block (32, LOAD_CHECK_WARPS): warp y checks list entry blockIdx.x * LOAD_CHECK_WARPS + y.
// The screen section is read as aligned 16-byte units; its words all start at the same byte of a 32-bit word (rows start at
// 2i mod 16), so each is a funnel shift of two loaded words.  An accepted entry claims its env with atomicMax of its key:
// of the accepted entries for one env, the last in the list holds the claim when the kernel ends.
__global__ void __launch_bounds__(32 * LOAD_CHECK_WARPS) k_load_check(const int32_t *__restrict__ ids, int n, int n_envs, const uint8_t *__restrict__ blobs,
                                                                      int32_t *__restrict__ status, unsigned long long *__restrict__ claim, uint32_t seq) {
    const int i = blockIdx.x * LOAD_CHECK_WARPS + threadIdx.y, lane = threadIdx.x;
    if (i >= n) return;
    const int env = ids ? ids[i] : i;
    if (env < 0 || env >= n_envs) {
        if (status && lane == 0) status[i] = GBENV_E_ARG;
        return;
    }
    const uint8_t *row = blobs + (size_t)i * GBENV_STATE_BYTES;
    bool ok = true;
    if (lane == 0) ok = state_head_ok(c_layout, [&](uint32_t o) { return (uint32_t)__ldg(row + o); });
    const StateSection &fb = c_layout.s[STATE_FB_SECTION];
    const size_t g0 = (size_t)i * GBENV_STATE_BYTES + fb.off, g1 = g0 + fb.len;  // screen bytes, from the aligned base
    const uint32_t sh = 8 * (uint32_t)(g0 & 3);
    const uint4 *units = reinterpret_cast<const uint4 *>(blobs);
    const uint32_t *words = reinterpret_cast<const uint32_t *>(blobs);
    for (size_t u = (g0 >> 4) + lane; u < (g1 + 15) >> 4; u += 32) {
        const uint4 q = __ldg(units + u);
        const uint32_t v[5] = {q.x, q.y, q.z, q.w, __ldg(words + 4 * u + 4)};  // the screen is followed by WRAM: still in the row
#pragma unroll
        for (int t = 0; t < 4; t++) {
            const size_t a = 16 * u + 4 * t + (g0 & 3);  // the screen word that starts in word t of the unit
            if (a >= g0 && a < g1) ok &= state_shade_ok(__funnelshift_r(v[t], v[t + 1], sh));
        }
    }
    ok = __all_sync(0xFFFFFFFFu, ok);
    if (lane == 0) {
        if (status) status[i] = ok ? GBENV_OK : GBENV_E_STATE;
        if (ok) atomicMax(claim + env, load_key(seq, i));
    }
}

// grid (ceil(n / 32), LOAD_PLAN.n_chunks), block (32, LOAD_WARPS).
// Staging: warp y takes entries y, y + 8, ..; its lanes read the chunk's windows of the entry's row as consecutive aligned
// 16-byte units into shared memory, one row per entry.  Writing: lane x takes entry x and warp y every LOAD_WARPS-th image
// word of the chunk, derived by state_image_word from the staged bytes (a file word is a funnel shift of two staged words)
// and stored through image_slot, so when the entries are the 32 envs of a tile in order each warp store is one 128-byte
// line.  Register words are merged with the env's old ones as a PyBoy v9 load does.  An entry whose env's claim is not its
// own key (out-of-range id, rejected row, or a later entry for the same env) stages and writes nothing.
__global__ void __launch_bounds__(GB_TILE * LOAD_WARPS) k_load_states(const DevArrays d, const int32_t *__restrict__ ids, int n, const uint8_t *__restrict__ blobs,
                                                                     const unsigned long long *__restrict__ claim, uint32_t seq) {
    __shared__ uint32_t s_img[GB_TILE * LOAD_ROW];
    __shared__ int s_env[GB_TILE];
    const int tx = threadIdx.x, ty = threadIdx.y, first = blockIdx.x * GB_TILE, c = blockIdx.y;
    const uint32_t win0 = c_lplan.win0[c], nwin = c_lplan.nwin[c];
    const size_t total = (size_t)n * GBENV_STATE_BYTES;
    if (ty == 0) {
        int env = -1;
        if (first + tx < n) {
            const int e = ids ? ids[first + tx] : first + tx;
            if (e >= 0 && e < d.n_envs && claim[e] == load_key(seq, first + tx)) env = e;
        }
        s_env[tx] = env;
    }
    __syncthreads();
    for (int k = ty; k < GB_TILE; k += LOAD_WARPS) {
        if (s_env[k] < 0) continue;
        const size_t row0 = (size_t)(first + k) * GBENV_STATE_BYTES;
        uint32_t *srow = s_img + k * LOAD_ROW;
        for (uint32_t m = 0; m < nwin; m++) {
            const size_t u0 = (row0 + c_lplan.lo[win0 + m]) >> 4, end = row0 + c_lplan.hi[win0 + m] + 3;
            const size_t u1 = ((end < total ? end : total) + 15) >> 4;
            for (size_t u = u0 + tx; u < u1; u += 32) {
                uint4 q;
                if (16 * u + 16 <= total) {
                    q = __ldg(reinterpret_cast<const uint4 *>(blobs) + u);
                } else {  // the last unit of the buffer, which may end inside it
                    uint32_t b[4] = {0, 0, 0, 0};
                    for (size_t x = 16 * u; x < total; x++) b[(x >> 2) & 3] |= (uint32_t)blobs[x] << (8 * (x & 3));
                    q = make_uint4(b[0], b[1], b[2], b[3]);
                }
                uint32_t *dst = srow + c_lplan.base[win0 + m] + 4 * (uint32_t)(u - u0);
                dst[0] = q.x; dst[1] = q.y; dst[2] = q.z; dst[3] = q.w;
            }
        }
    }
    __syncthreads();
    const int env = s_env[tx];
    if (env < 0) return;
    const size_t row0 = (size_t)(first + tx) * GBENV_STATE_BYTES;
    const uint32_t *srow = s_img + tx * LOAD_ROW;
    const auto rd = [&](uint32_t o) -> uint32_t {
        uint32_t m = 0;
        while (m + 1 < nwin && c_lplan.lo[win0 + m + 1] <= o) m++;
        const size_t g = row0 + o;
        const uint32_t w = c_lplan.base[win0 + m] + (uint32_t)((g >> 2) - (((row0 + c_lplan.lo[win0 + m]) >> 4) << 2));
        return __funnelshift_r(srow[w], srow[w + 1], 8 * (uint32_t)(g & 3));
    };
    const uint32_t seg0 = c_lplan.seg0[c], nseg = c_lplan.nseg[c];
    for (uint32_t sg = seg0; sg < seg0 + nseg; sg++) {
        const uint64_t secs = c_lplan.secs[sg];
        for (uint32_t j = c_lplan.j0[sg] + ty; j < c_lplan.j1[sg]; j += LOAD_WARPS) {
            uint32_t v = state_image_word(c_layout, secs, j, rd);
            uint32_t *slot = image_slot(d, env, j);
            if (j >= IMG_REGS) v = merge_loaded_reg(j - IMG_REGS, *slot, v, 9, rd(STATE_OFF_LCDC) & 0xFF);
            *slot = v;
        }
    }
}

cudaError_t launch_load_states(const DevArrays &d, const int32_t *ids, int n, const uint8_t *blobs, int32_t *status, unsigned long long *claim,
                               uint32_t seq, cudaStream_t st) {
    k_load_check<<<(n + LOAD_CHECK_WARPS - 1) / LOAD_CHECK_WARPS, dim3(32, LOAD_CHECK_WARPS), 0, st>>>(ids, n, d.n_envs, blobs, status, claim, seq);
    k_load_states<<<dim3((n + GB_TILE - 1) / GB_TILE, LOAD_PLAN.n_chunks), dim3(GB_TILE, LOAD_WARPS), 0, st>>>(d, ids, n, blobs, claim, seq);
    return cudaGetLastError();
}
