// gb_events.cu -- the event flags of a list of envs (gbenv_event_flags), linked into libgbenv.so next to gbenv.cu.
//
// Entry k of the event table (event_bits.inc) is bit k & 31 of word k >> 5 of an env's row; bits 130..159 are 0.  The flags
// sit in plain WRAM (0xD765-0xD838), whose byte i of env e is byte i & 3 of word il_index(e / 32, MEM_WORDS, i / 4, e % 32).
#include <stdint.h>
#include "../../include/gbenv.h"
#include "gb_events.cuh"
#include "gb_layout.cuh"

#define EVENT_THREADS 128

// address | bit << 16 of every table entry.  Internal linkage (c_events of gb_wrap.cuh is the same table with weights for the
// step's rewards); a constant the compiler sees, so the loop below unrolls into loads at fixed offsets.
#define EV(a, b, w) ((uint32_t)(a) | ((uint32_t)(b) << 16))
static __device__ const uint32_t c_event_bits[GBENV_EVENT_FLAGS] = {
#include "event_bits.inc"
};
#undef EV
static_assert(GBENV_EVENT_WORDS * 32 >= GBENV_EVENT_FLAGS, "a row holds every flag");

__device__ __forceinline__ uint32_t wram_word_of(uint32_t addr) { return (MEM_WRAM + (addr - 0xC000u)) >> 2; }

// One thread per list entry: lane x of a warp takes entry x, so when the entries are the 32 envs of one tile in order (NULL
// ids) every load of the warp is one whole 128-byte line.  Each WRAM word the table touches is loaded once (the compiler
// merges the table's repeated loads of a word; 17 distinct words), all loads are issued before the bits are assembled, and
// the row leaves in GBENV_EVENT_WORDS plain stores: a warp's stores cover 640 contiguous bytes.
__global__ void __launch_bounds__(EVENT_THREADS) k_event_flags(const uint32_t *__restrict__ mem, const int32_t *__restrict__ ids, int n,
                                                               int n_envs, uint32_t *__restrict__ flags) {
    const int i = blockIdx.x * EVENT_THREADS + threadIdx.x;
    if (i >= n) return;
    const int env = ids ? ids[i] : i;
    if (env < 0 || env >= n_envs) return;
    const uint32_t *src = mem + il_index(env >> 5, MEM_WORDS, 0, env & 31);
    uint32_t row[GBENV_EVENT_WORDS] = {};
#pragma unroll
    for (int k = 0; k < GBENV_EVENT_FLAGS; k++) {
        const uint32_t a = c_event_bits[k] & 0xFFFF, b = c_event_bits[k] >> 16;
        const uint32_t word = __ldg(src + (size_t)wram_word_of(a) * GB_TILE);
        row[k >> 5] |= ((word >> (8 * (a & 3) + b)) & 1u) << (k & 31);
    }
    uint32_t *dst = flags + (size_t)i * GBENV_EVENT_WORDS;
#pragma unroll
    for (int w = 0; w < GBENV_EVENT_WORDS; w++) dst[w] = row[w];
}

cudaError_t launch_event_flags(const uint32_t *mem, const int32_t *ids, int n, int n_envs, uint32_t *flags, cudaStream_t st) {
    k_event_flags<<<(n + EVENT_THREADS - 1) / EVENT_THREADS, EVENT_THREADS, 0, st>>>(mem, ids, n, n_envs, flags);
    return cudaGetLastError();
}
