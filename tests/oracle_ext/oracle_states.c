/*
 * tests/oracle_ext/oracle_states.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * gbenv_save_states of include/gbenv.h for the CPU oracle, prefixed `oracle_`, all pointers host memory.  Linked into
 * liboracle.so next to oracle/oracle_api.c (__graft_entry__.build_oracle) and written only against that file's exported
 * entry points (oracle_save_state, oracle_num_envs), so the oracle's own sources stay as they are.
 */
#include <stdint.h>

#include "../../include/gbenv.h"

typedef struct oracle oracle;
int oracle_num_envs(const oracle *h);
int oracle_save_state(oracle *h, int env, uint8_t *blob);

int oracle_save_states(oracle *h, const int32_t *env_ids, int n, uint8_t *blobs, void *stream) {
    (void)stream;
    if (!h || n < 0 || (!env_ids && n > oracle_num_envs(h)) || (n && (!blobs || ((uintptr_t)blobs & 15)))) return GBENV_E_ARG;
    for (int i = 0; i < n; i++) {
        const int env = env_ids ? env_ids[i] : i;
        if (env < 0 || env >= oracle_num_envs(h)) continue; /* row left untouched */
        const int rc = oracle_save_state(h, env, blobs + (size_t)i * GBENV_STATE_BYTES);
        if (rc != GBENV_OK) return rc;
    }
    return GBENV_OK;
}
