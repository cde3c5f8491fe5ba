/*
 * tests/oracle_ext/oracle_obs.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The packed-observation calls of include/gbenv.h (gbenv_step_packed, gbenv_reset_packed, gbenv_unpack_obs) for the CPU
 * oracle, prefixed `oracle_`, all pointers host memory.  Linked into liboracle.so next to oracle/oracle_api.c
 * (__graft_entry__.build_oracle) and written only against that file's exported entry points: the step and reset write the
 * reference observation into a scratch buffer through oracle_step_masked / oracle_reset_dev, and pack() below turns the rows
 * they wrote into the packed layout.  pack() is the CPU reference of that layout; it refuses an observation outside it (a
 * grey that is not one of the four levels, channels 0-2 that differ, channel 3 not 0 or 255).
 */
#include <stdint.h>
#include <stdlib.h>

#include "../../include/gbenv.h"

typedef struct oracle oracle;
int oracle_num_envs(const oracle *h);
int oracle_step_masked(oracle *h, const uint8_t *actions, const uint8_t *skip, uint8_t *obs, size_t obs_stride, double *reward, uint8_t *done,
                       void *stream);
int oracle_reset_dev(oracle *h, const uint8_t *mask, int max_episode_steps, double reward_scale, uint8_t *obs, size_t obs_stride, void *stream);

static const uint8_t GREY[4] = {0xFF, 0x99, 0x55, 0x00};

static int misaligned(const void *p) { return ((uintptr_t)p & 15) != 0; }

/* one env's reference observation -> its GBENV_OBS_PACKED_WORDS words */
static int pack(const uint8_t *obs, uint32_t *row) {
    for (int w = 0; w < GBENV_OBS_PACKED_WORDS; w++) row[w] = 0;
    for (int i = 0; i < GBENV_OBS_H; i++) {
        for (int j = 0; j < GBENV_OBS_W; j++) {
            const uint8_t *px = obs + (i * GBENV_OBS_W + j) * GBENV_OBS_C;
            int s = 0;
            while (s < 4 && GREY[s] != px[0]) s++;
            if (s == 4 || px[1] != px[0] || px[2] != px[0] || (px[3] != 0 && px[3] != 255)) return GBENV_E_STATE;
            row[8 * i + j / 16] |= (uint32_t)s << (2 * (j & 15));
            if (px[3]) row[8 * i + 5 + j / 32] |= 1u << (j & 31);
        }
    }
    return GBENV_OK;
}

/* pack the rows of the envs whose byte in `sel` equals `want` (sel NULL: all) from the scratch observations */
static int pack_rows(oracle *h, const uint8_t *scratch, const uint8_t *sel, int want, uint32_t *packed) {
    for (int e = 0; e < oracle_num_envs(h); e++) {
        if (sel && (sel[e] != 0) != want) continue;
        int rc = pack(scratch + (size_t)e * GBENV_OBS_BYTES, packed + (size_t)e * GBENV_OBS_PACKED_WORDS);
        if (rc) return rc;
    }
    return GBENV_OK;
}

int oracle_step_packed(oracle *h, const uint8_t *actions, const uint8_t *skip, uint32_t *packed, double *reward, uint8_t *done, void *stream) {
    if (!h || !actions || !packed || !reward || !done || misaligned(packed)) return GBENV_E_ARG;
    uint8_t *scratch = (uint8_t *)calloc((size_t)oracle_num_envs(h), GBENV_OBS_BYTES);
    if (!scratch) return GBENV_E_NOMEM;
    int rc = oracle_step_masked(h, actions, skip, scratch, GBENV_OBS_BYTES, reward, done, stream);
    if (rc == GBENV_OK) rc = pack_rows(h, scratch, skip, 0, packed);
    free(scratch);
    return rc;
}

int oracle_reset_packed(oracle *h, const uint8_t *mask, int max_episode_steps, double reward_scale, uint32_t *packed, void *stream) {
    if (!h || !packed || misaligned(packed)) return GBENV_E_ARG;
    uint8_t *scratch = (uint8_t *)calloc((size_t)oracle_num_envs(h), GBENV_OBS_BYTES);
    if (!scratch) return GBENV_E_NOMEM;
    int rc = oracle_reset_dev(h, mask, max_episode_steps, reward_scale, scratch, GBENV_OBS_BYTES, stream);
    if (rc == GBENV_OK) rc = pack_rows(h, scratch, mask, 1, packed);
    free(scratch);
    return rc;
}

int oracle_unpack_obs(oracle *h, const uint32_t *packed, int n, uint8_t *out, void *stream) {
    (void)stream;
    if (!h || n < 0 || (n && (!packed || !out)) || misaligned(packed) || misaligned(out)) return GBENV_E_ARG;
    for (size_t e = 0; e < (size_t)n; e++) {
        const uint32_t *row = packed + e * GBENV_OBS_PACKED_WORDS;
        uint8_t *obs = out + e * GBENV_OBS_BYTES;
        for (int i = 0; i < GBENV_OBS_H; i++) {
            for (int j = 0; j < GBENV_OBS_W; j++) {
                uint8_t *px = obs + (i * GBENV_OBS_W + j) * GBENV_OBS_C;
                px[0] = px[1] = px[2] = GREY[(row[8 * i + j / 16] >> (2 * (j & 15))) & 3];
                px[3] = (row[8 * i + 5 + j / 32] >> (j & 31)) & 1 ? 255 : 0;
            }
        }
    }
    return GBENV_OK;
}
