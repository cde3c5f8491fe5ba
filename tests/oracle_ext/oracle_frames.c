/*
 * tests/oracle_ext/oracle_frames.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The batched frame calls of include/gbenv.h (gbenv_capture_frames, gbenv_frames_to_rgb) for the CPU oracle, prefixed
 * `oracle_`, all pointers host memory.  Linked into liboracle.so next to oracle/oracle_api.c (__graft_entry__.build_oracle)
 * and written only against that file's exported entry points: the packed frame is rebuilt from oracle_screen's RGB, whose
 * grey level names the shade, so the oracle's own sources stay as they are.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/gbenv.h"

typedef struct oracle oracle;
int oracle_num_envs(const oracle *h);
int oracle_screen(oracle *h, int env, uint8_t *rgb);

#define PIXELS (GBENV_SCREEN_H * GBENV_SCREEN_W)

static const uint8_t GREY[4] = {0xFF, 0x99, 0x55, 0x00};

int oracle_capture_frames(oracle *h, const int32_t *env_ids, int n, uint32_t *frames, void *stream) {
    (void)stream;
    if (!h || n < 0 || (!env_ids && n > oracle_num_envs(h)) || (n && !frames)) return GBENV_E_ARG;
    uint8_t *rgb = (uint8_t *)malloc(3 * PIXELS);
    if (!rgb) return GBENV_E_NOMEM;
    int rc = GBENV_OK;
    for (int i = 0; i < n && rc == GBENV_OK; i++) {
        const int env = env_ids ? env_ids[i] : i;
        if (env < 0 || env >= oracle_num_envs(h)) continue;  // row left untouched
        rc = oracle_screen(h, env, rgb);
        uint32_t *row = frames + (size_t)i * GBENV_FRAME_WORDS;
        memset(row, 0, sizeof(uint32_t) * GBENV_FRAME_WORDS);
        for (int p = 0; rc == GBENV_OK && p < PIXELS; p++) {
            int s = 0;
            while (s < 4 && GREY[s] != rgb[3 * p]) s++;
            if (s == 4) rc = GBENV_E_STATE;  // not one of the four DMG greys
            else row[p >> 4] |= (uint32_t)s << (2 * (p & 15));
        }
    }
    free(rgb);
    return rc;
}

int oracle_frames_to_rgb(oracle *h, const uint32_t *frames, int n_frames, int channels, uint8_t *out, void *stream) {
    (void)stream;
    if (!h || n_frames < 0 || (channels != 1 && channels != 3) || (n_frames && (!frames || !out))) return GBENV_E_ARG;
    for (size_t p = 0; p < (size_t)n_frames * PIXELS; p++) {
        const uint8_t g = GREY[(frames[p >> 4] >> (2 * (p & 15))) & 3];
        for (int c = 0; c < channels; c++) out[p * channels + c] = g;
    }
    return GBENV_OK;
}
