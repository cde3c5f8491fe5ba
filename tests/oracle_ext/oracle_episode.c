/*
 * tests/oracle_ext/oracle_episode.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The episode-end reductions of include/gbenv.h (gbenv_counts_map_sum, gbenv_reduce_info_masked) for the CPU oracle,
 * prefixed `oracle_`, all pointers host memory.  Linked into liboracle.so next to oracle/oracle_api.c
 * (__graft_entry__.build_oracle) and written only against that file's exported entry points, so the oracle's own
 * sources stay as they are.
 */
#include <stdlib.h>
#include <string.h>

#include "../../include/gbenv.h"

typedef struct oracle oracle;
int oracle_num_envs(const oracle *h);
int oracle_get_info(oracle *h, double *info, void *stream);
int oracle_counts_map(oracle *h, int env, int32_t *map);

#define MAP_CELLS (444 * 436)

/* Same arithmetic as oracle_reduce_info (rows added env by env, slot by slot), over the masked envs only, so a NULL mask
 * gives its result bit for bit. */
int oracle_reduce_info_masked(oracle *h, const uint8_t *mask, double *sum, void *stream) {
    if (!h || !sum) return GBENV_E_ARG;
    const int n = oracle_num_envs(h);
    double *rows = (double *)malloc(sizeof(double) * GBENV_INFO_SCALARS * (size_t)n);
    if (!rows) return GBENV_E_NOMEM;
    int rc = oracle_get_info(h, rows, stream);
    if (rc == GBENV_OK) {
        memset(sum, 0, sizeof(double) * GBENV_INFO_SCALARS);
        for (int e = 0; e < n; e++) {
            if (mask && !mask[e]) continue;
            for (int k = 0; k < GBENV_INFO_SCALARS; k++) sum[k] += rows[(size_t)e * GBENV_INFO_SCALARS + k];
        }
    }
    free(rows);
    return rc;
}

/* int64 sum of the heat maps of the masked envs (-1 marks included), sum overwritten. */
int oracle_counts_map_sum(oracle *h, const uint8_t *mask, int64_t *sum, void *stream) {
    (void)stream;
    if (!h || !sum) return GBENV_E_ARG;
    int32_t *map = (int32_t *)malloc(sizeof(int32_t) * MAP_CELLS);
    if (!map) return GBENV_E_NOMEM;
    memset(sum, 0, sizeof(int64_t) * MAP_CELLS);
    int rc = GBENV_OK;
    for (int e = 0, n = oracle_num_envs(h); e < n && rc == GBENV_OK; e++) {
        if (mask && !mask[e]) continue;
        rc = oracle_counts_map(h, e, map);
        for (int i = 0; rc == GBENV_OK && i < MAP_CELLS; i++) sum[i] += map[i];
    }
    free(map);
    return rc;
}
