// load_table.cpp -- TEST INFRASTRUCTURE ONLY: the table-driven v9 parser and validity rules of
// pokegym_b200/csrc/gb_image.h that k_load_states runs (state_image_word, state_row_valid), next to the hand-written parser
// blob_to_image, compiled by g++ (-DGB_HOSTSIM, see gb_hd.h) for tests/test_load_states_cpu.py.
#define GB_HOSTSIM 1
#include "../../pokegym_b200/csrc/gb_hd.h"
#include "../../pokegym_b200/csrc/gb_image.h"

// file bytes o .. o + 3 of a v9 row as a little-endian word (bytes past the end read as 0)
static uint32_t st_rd(const uint8_t *row, uint32_t o) {
    uint32_t v = 0;
    for (uint32_t k = 0; k < 4 && o + k < GBENV_STATE_BYTES; k++) v |= (uint32_t)row[o + k] << (8 * k);
    return v;
}

extern "C" {

// v9 row -> canonical image (IMG_WORDS words) through the table (state_image_word, every section offered for every word)
void st_image_from_row(const uint8_t *row, uint32_t *img) {
    const auto rd = [row](uint32_t o) { return st_rd(row, o); };
    for (uint32_t j = 0; j < IMG_WORDS; j++) img[j] = state_image_word(STATE_LAYOUT, (1ull << STATE_SECTIONS) - 1, j, rd);
}

// the same through the hand-written parser; 0 or its error
int st_blob_to_image(const uint8_t *blob, size_t len, uint32_t *img) {
    std::vector<uint32_t> v;
    int ver = 0;
    std::string err;
    const int rc = blob_to_image(blob, len, v, &ver, err);
    if (rc == 0) memcpy(img, v.data(), IMG_WORDS * sizeof(uint32_t));
    return rc;
}

// state_row_valid: 1 when the row is a loadable v9 file
int st_row_valid(const uint8_t *row) { return state_row_valid(STATE_LAYOUT, [row](uint32_t o) { return st_rd(row, o); }) ? 1 : 0; }

int st_img_words(void) { return IMG_WORDS; }
}
