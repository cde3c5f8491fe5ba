/*
 * tests/oracle_ext/oracle_events.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * gbenv_event_flags of include/gbenv.h for the CPU oracle, prefixed `oracle_`, all pointers host memory.  Linked into
 * liboracle.so next to oracle/oracle_api.c (__graft_entry__.build_oracle) and written only against that file's exported
 * entry points (oracle_read_mem, oracle_num_envs), so the oracle's own sources stay as they are.  The table is the same
 * file the CUDA kernels include.
 */
#include <stdint.h>
#include <string.h>

#include "../../include/gbenv.h"

typedef struct oracle oracle;
int oracle_num_envs(const oracle *h);
int oracle_read_mem(oracle *h, int env, uint32_t addr, uint32_t n, uint8_t *out);

typedef struct {
    uint16_t addr, bit;
    int weight;
} event_bit;

#define EV(a, b, w) {a, b, w}
static const event_bit EVENTS[] = {
#include "../../pokegym_b200/csrc/event_bits.inc"
};
#undef EV

_Static_assert(sizeof(EVENTS) / sizeof(EVENTS[0]) == GBENV_EVENT_FLAGS, "one entry per event flag");

#define LO 0xD700u /* every table address lies in [LO, LO + SPAN) */
#define SPAN 0x200u

int oracle_event_flags(oracle *h, const int32_t *env_ids, int n, uint32_t *flags, void *stream) {
    (void)stream;
    if (!h || n < 0 || (!env_ids && n > oracle_num_envs(h)) || (n && !flags)) return GBENV_E_ARG;
    uint8_t wram[SPAN];
    for (int i = 0; i < n; i++) {
        const int env = env_ids ? env_ids[i] : i;
        if (env < 0 || env >= oracle_num_envs(h)) continue; /* row left untouched */
        const int rc = oracle_read_mem(h, env, LO, SPAN, wram);
        if (rc != GBENV_OK) return rc;
        uint32_t *row = flags + (size_t)i * GBENV_EVENT_WORDS;
        memset(row, 0, sizeof(uint32_t) * GBENV_EVENT_WORDS);
        for (int k = 0; k < GBENV_EVENT_FLAGS; k++)
            row[k >> 5] |= (uint32_t)((wram[EVENTS[k].addr - LO] >> EVENTS[k].bit) & 1) << (k & 31);
    }
    return GBENV_OK;
}
