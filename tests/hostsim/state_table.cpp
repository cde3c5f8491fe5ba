// state_table.cpp -- TEST INFRASTRUCTURE ONLY: the v9 section table of pokegym_b200/csrc/gb_image.h (STATE_LAYOUT), and the
// host serialiser built on it, compiled by g++ (-DGB_HOSTSIM, see gb_hd.h) for tests/test_save_states_cpu.py.
#define GB_HOSTSIM 1
#include "../../pokegym_b200/csrc/gb_hd.h"
#include "../../pokegym_b200/csrc/gb_image.h"

extern "C" {

// off, len, src, kind, shift, mask of every section, in file order; returns the section count
int st_sections(uint32_t *out) {
    for (int i = 0; i < STATE_SECTIONS; i++) {
        const StateSection &s = STATE_LAYOUT.s[i];
        const uint32_t row[6] = {s.off, s.len, s.src, s.kind, s.shift, s.mask};
        for (int k = 0; k < 6; k++) out[6 * i + k] = row[k];
    }
    return STATE_SECTIONS;
}

// index of the section holding file byte o
int st_section_of(uint32_t o) { return state_section_of(STATE_LAYOUT, o); }

// blob -> canonical image (blob_to_image) -> v9 file (image_to_blob, i.e. the section table); 0 or the parser's error
int st_roundtrip(const uint8_t *blob, size_t len, uint8_t *out) {
    std::vector<uint32_t> img;
    int ver = 0;
    std::string err;
    const int rc = blob_to_image(blob, len, img, &ver, err);
    if (rc) return rc;
    image_to_blob(img, out);
    return 0;
}
}
