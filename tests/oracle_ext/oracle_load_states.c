/*
 * tests/oracle_ext/oracle_load_states.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * gbenv_load_states of include/gbenv.h for the CPU oracle, prefixed `oracle_`, all pointers host memory.  Linked into
 * liboracle.so next to oracle/oracle_api.c (__graft_entry__.build_oracle) and written only against that file's exported
 * entry points (oracle_add_state_template, oracle_load_template, oracle_num_envs), so the oracle's own sources stay as they
 * are.
 */
#include <stdint.h>
#include <stdlib.h>

#include "../../include/gbenv.h"

typedef struct oracle oracle;
int oracle_num_envs(const oracle *h);
int oracle_add_state_template(oracle *h, const uint8_t *blob, size_t len, int *id_out);
int oracle_load_template(oracle *h, const int32_t *ids, int n, int t);

/* The v9 offsets the acceptance rules read (SURVEY.md 8c), written out here rather than taken from the CUDA library's
 * section table, so that the rules are checked against an independent statement of them. */
#define V9_CGB 4             /* header: bootrom_enabled, key1, double_speed, cgb */
#define V9_CLOCK_HIGH 8392   /* high 32 bits of the u64 clock at 8388 */
#define V9_TARGET_HIGH 8400  /* high 32 bits of the u64 clock_target at 8396 */
#define V9_SCREEN 9125       /* 144 x 160 little-endian PyBoy words */
#define V9_SCREEN_WORDS (144 * 160)

static int v9_loadable(const uint8_t *b) {
    static const uint32_t shades[4] = {0xFFFFFF01u, 0x99999900u, 0x55555500u, 0x00000000u};
    if (b[0] != 9 || b[V9_CGB] != 0) return 0;
    for (int k = 0; k < 4; k++)
        if (b[V9_CLOCK_HIGH + k] || b[V9_TARGET_HIGH + k]) return 0;
    for (int i = 0; i < V9_SCREEN_WORDS; i++) {
        const uint8_t *p = b + V9_SCREEN + 4 * i;
        const uint32_t w = p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
        if (w != shades[0] && w != shades[1] && w != shades[2] && w != shades[3]) return 0;
    }
    return 1;
}

/* Entry i: env env_ids[i] (NULL: i) from row i.  Out-of-range ids are skipped (status GBENV_E_ARG), rows that are not
 * loadable v9 files rejected (GBENV_E_STATE); of the accepted entries for one env the last is loaded, through a template
 * (which the oracle keeps: this is test infrastructure). */
int oracle_load_states(oracle *h, const int32_t *env_ids, int n, const uint8_t *blobs, int32_t *status, void *stream) {
    (void)stream;
    if (!h || n < 0 || (!env_ids && n > oracle_num_envs(h)) || (n && (!blobs || ((uintptr_t)blobs & 15))) || ((uintptr_t)env_ids & 3) ||
        ((uintptr_t)status & 3))
        return GBENV_E_ARG;
    const int n_envs = oracle_num_envs(h);
    int *last = (int *)malloc(sizeof(int) * (size_t)n_envs);
    for (int e = 0; e < n_envs; e++) last[e] = -1;
    for (int i = 0; i < n; i++) {
        const int env = env_ids ? env_ids[i] : i;
        int st = GBENV_E_ARG;
        if (env >= 0 && env < n_envs) {
            st = v9_loadable(blobs + (size_t)i * GBENV_STATE_BYTES) ? GBENV_OK : GBENV_E_STATE;
            if (st == GBENV_OK) last[env] = i;
        }
        if (status) status[i] = st;
    }
    int rc = GBENV_OK;
    for (int i = 0; i < n && rc == GBENV_OK; i++) {
        const int32_t env = env_ids ? env_ids[i] : i;
        if (env < 0 || env >= n_envs || last[env] != i) continue;
        int tid = -1;
        rc = oracle_add_state_template(h, blobs + (size_t)i * GBENV_STATE_BYTES, GBENV_STATE_BYTES, &tid);
        if (rc == GBENV_OK) rc = oracle_load_template(h, &env, 1, tid);
    }
    free(last);
    return rc;
}
