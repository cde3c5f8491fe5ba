// gb_image.h -- PyBoy save-state blob <-> canonical per-env image (host code), and the v9 section table the device
// serialiser shares.
//
// The canonical image is the linear word layout of gb_layout.cuh (IMG_*): what state templates hold on the device and
// what k_scatter_image / k_gather_image move in and out of the interleaved arrays.  Shared by libgbenv.so (gbenv.cu)
// and the host-simulation test harness (tests/hostsim).
// Replaces pyboy_binding.open_state_file / load_pyboy_state (/root/reference/pokegym/pyboy_binding.py:59-69) and
// PyBoy.save_state; the field order is SURVEY.md section 8c.
#pragma once
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/gbenv.h"
#include "gb_layout.cuh"

static inline void img_set_byte(std::vector<uint32_t> &img, uint32_t base_word, uint32_t byte_index, uint8_t v) {
    uint32_t &w = img[base_word + (byte_index >> 2)];
    uint32_t sh = (byte_index & 3) * 8;
    w = (w & ~(0xFFu << sh)) | ((uint32_t)v << sh);
}
static inline uint8_t img_get_byte(const std::vector<uint32_t> &img, uint32_t base_word, uint32_t byte_index) {
    return (uint8_t)(img[base_word + (byte_index >> 2)] >> ((byte_index & 3) * 8));
}

static const uint32_t SHADE_WORDS[4] = {0xFFFFFF01u, 0x99999900u, 0x55555500u, 0x00000000u};

// ---- The PyBoy v9 file as a table of sections over the canonical image (SURVEY.md 8c).  This is the one definition of the
// v9 layout on the C++ side: image_to_blob (host; also tests/hostsim) and k_save_states (gb_state.cu) both serialise from
// it.  A section is a run of file bytes [off, off + len) with one source:
//   SK_CONST  every byte is `src`
//   SK_FIELD  one byte, (image word src >> shift) & mask  (the flag bits of R_INT, next_stat_mode)
//   SK_BYTES  image bytes src .. src + len - 1, image byte i being byte i & 3 of image word i >> 2 (RAM, register bytes)
//   SK_LP     144 scanline records of 5 bytes: the 4 bytes of IMG_LP word 2y, then bit 4 of word 2y + 1
//   SK_FB     one PyBoy word per pixel, little-endian: SHADE_WORDS of the 2-bit shade, 16 pixels per IMG_FB word
enum : uint8_t { SK_CONST, SK_FIELD, SK_BYTES, SK_LP, SK_FB };
struct StateSection {
    uint32_t off, len, src;
    uint8_t kind, shift, mask;
};
#define STATE_SECTIONS 42
struct StateLayout {
    StateSection s[STATE_SECTIONS];
};

constexpr uint32_t state_reg_byte(uint32_t r, uint32_t byte) { return (IMG_REGS + r) * 4u + byte; }

constexpr StateLayout make_state_layout() {
    StateLayout t{};
    uint32_t off = 0;
    int i = 0;
    struct Add {
        StateLayout &t;
        uint32_t &off;
        int &i;
        constexpr void operator()(uint8_t kind, uint32_t len, uint32_t src, uint8_t shift = 0, uint8_t mask = 0xFF) {
            t.s[i].off = off; t.s[i].len = len; t.s[i].src = src; t.s[i].kind = kind; t.s[i].shift = shift; t.s[i].mask = mask;
            off += len;
            i++;
        }
    } add{t, off, i};
    add(SK_CONST, 1, 9);                                  // version
    add(SK_BYTES, 4, state_reg_byte(R_HDR, 0));           // bootrom_enabled, key1, double_speed, cgb
    add(SK_BYTES, 2, state_reg_byte(R_HLAF, 2));          // A F
    add(SK_BYTES, 1, state_reg_byte(R_BCDE, 1));          // B
    add(SK_BYTES, 1, state_reg_byte(R_BCDE, 0));          // C
    add(SK_BYTES, 1, state_reg_byte(R_BCDE, 3));          // D
    add(SK_BYTES, 1, state_reg_byte(R_BCDE, 2));          // E
    add(SK_BYTES, 2, state_reg_byte(R_HLAF, 0));          // HL
    add(SK_BYTES, 4, state_reg_byte(R_SPPC, 0));          // SP PC
    add(SK_FIELD, 1, IMG_REGS + R_INT, 0, 1);             // IME
    add(SK_FIELD, 1, IMG_REGS + R_INT, 1, 1);             // halted
    add(SK_FIELD, 1, IMG_REGS + R_INT, 2, 1);             // stopped
    add(SK_BYTES, 1, state_reg_byte(R_INT, 1));           // IE
    add(SK_FIELD, 1, IMG_REGS + R_INT, 3, 1);             // interrupt_queued
    add(SK_BYTES, 1, state_reg_byte(R_INT, 2));           // IF
    add(SK_BYTES, 0x2000, IMG_MEM * 4 + MEM_VRAM);        // VRAM
    add(SK_BYTES, 0xA0, IMG_MEM * 4 + MEM_HI);            // OAM
    add(SK_BYTES, 1, state_reg_byte(R_LCD0, 0));          // LCDC
    add(SK_BYTES, 3, state_reg_byte(R_LCD2, 0));          // BGP OBP0 OBP1
    add(SK_BYTES, 3, state_reg_byte(R_LCD0, 1));          // STAT LY LYC
    add(SK_BYTES, 4, state_reg_byte(R_LCD1, 0));          // SCY SCX WY WX
    add(SK_BYTES, 1, state_reg_byte(R_HDR, 3));           // cgb
    add(SK_BYTES, 1, state_reg_byte(R_HDR, 2));           // double_speed
    add(SK_BYTES, 4, state_reg_byte(R_CLOCK, 0));         // clock (u64; the emulator keeps 32 bits)
    add(SK_CONST, 4, 0);
    add(SK_BYTES, 4, state_reg_byte(R_TARGET, 0));        // clock_target (u64)
    add(SK_CONST, 4, 0);
    add(SK_FIELD, 1, IMG_REGS + R_LCD2, 26, 3);           // next_stat_mode
    add(SK_LP, 144 * 5, IMG_LP);                          // scanline parameters
    add(SK_FB, 144 * 160 * 4, IMG_FB);                    // screen
    add(SK_BYTES, 0x2000, IMG_MEM * 4 + MEM_WRAM);        // WRAM
    add(SK_BYTES, 96, IMG_MEM * 4 + MEM_HI + 0xA0);       // FEA0-FEFF
    add(SK_BYTES, 76, IMG_MEM * 4 + MEM_HI + 0x100);      // IO FF00-FF4B
    add(SK_BYTES, 127, IMG_MEM * 4 + MEM_HI + 0x180);     // HRAM
    add(SK_BYTES, 52, IMG_MEM * 4 + MEM_HI + 0x14C);      // FF4C-FF7F
    add(SK_BYTES, 2, state_reg_byte(R_TIMER, 0));         // DIV TIMA
    add(SK_BYTES, 2, state_reg_byte(R_DIVC, 0));          // DIV_counter (u16)
    add(SK_BYTES, 2, state_reg_byte(R_TIMAC, 0));         // TIMA_counter (u16)
    add(SK_BYTES, 2, state_reg_byte(R_TIMER, 2));         // TMA TAC
    add(SK_BYTES, 4, state_reg_byte(R_MBC, 0));           // rombank rambank ram_enabled memorymodel
    add(SK_BYTES, CRAM_BYTES, IMG_CRAM * 4);              // cartridge RAM
    add(SK_BYTES, 2, state_reg_byte(R_JOY, 0));           // joypad directional, standard
    return t;
}

static constexpr StateLayout STATE_LAYOUT = make_state_layout();
static_assert(STATE_LAYOUT.s[STATE_SECTIONS - 1].off + STATE_LAYOUT.s[STATE_SECTIONS - 1].len == GBENV_STATE_BYTES, "v9 file length");
static_assert(STATE_LAYOUT.s[15].off == 23 && STATE_LAYOUT.s[30].off == 101285, "VRAM and WRAM offsets (SURVEY.md 8c)");

// the PyBoy framebuffer word of shade s (SHADE_WORDS[s]): grey in bytes 1..3, the colour-0 flag byte set for white
__host__ __device__ inline uint32_t state_shade_word(uint32_t s) { return ((0x005599FFu >> (8 * s)) & 0xFF) * 0x01010100u | (s == 0); }

// the image word file byte o (inside section s, which is not SK_CONST) is taken from
__host__ __device__ constexpr uint32_t state_word(const StateSection &s, uint32_t o) {
    const uint32_t r = o - s.off;
    return s.kind == SK_FIELD ? s.src
         : s.kind == SK_BYTES ? (s.src + r) >> 2
         : s.kind == SK_LP    ? IMG_LP + 2 * (r / 5) + (r % 5 == 4)
                              : IMG_FB + (r >> 6);
}
// file byte o (inside section s) given w = image word state_word(s, o) (ignored for SK_CONST)
__host__ __device__ inline uint8_t state_byte(const StateSection &s, uint32_t o, uint32_t w) {
    const uint32_t r = o - s.off;
    switch (s.kind) {
    case SK_CONST: return (uint8_t)s.src;
    case SK_FIELD: return (uint8_t)((w >> s.shift) & s.mask);
    case SK_BYTES: return (uint8_t)(w >> (8 * ((s.src + r) & 3)));
    case SK_LP: return (uint8_t)(r % 5 == 4 ? (w >> 4) & 1 : w >> (8 * (r % 5)));
    default: return (uint8_t)(state_shade_word((w >> (2 * ((r >> 2) & 15))) & 3) >> (8 * (r & 3)));
    }
}
// index of the section that holds file byte o
__host__ __device__ constexpr int state_section_of(const StateLayout &t, uint32_t o) {
    int lo = 0, hi = STATE_SECTIONS - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (t.s[mid].off <= o) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---- The other direction, v9 file -> canonical image, from the same table: state_image_word is the inverse of state_word /
// state_byte (k_load_states in gb_state.cu; tests/hostsim checks it against blob_to_image).

// Image bits a v9 file does not carry, the one definition blob_to_image and state_image_word share: R_JOY's ly_window
// (0xFF; a load keeps the env's own) and lp_dirty (144), R_MISC (0xFF: blank shade unknown, no lines pending), and R_LCD2's
// stat_mode bits, STAT & 3 (a load keeps the env's own).  R_INT's fault bit is 0, like every other bit not listed here.
__host__ __device__ constexpr uint32_t state_unfiled_bits(uint32_t j, uint32_t stat) {
    return j == IMG_REGS + R_JOY ? (0xFFu << 16) | (144u << 24) : j == IMG_REGS + R_MISC ? 0xFFu : j == IMG_REGS + R_LCD2 ? (stat & 3) << 24 : 0u;
}

// the file byte that holds image byte b; where the file holds a byte twice (double_speed, cgb) the first copy, which is the
// one blob_to_image reads
constexpr uint32_t state_file_byte(const StateLayout &t, uint32_t b) {
    for (int i = 0; i < STATE_SECTIONS; i++)
        if (t.s[i].kind == SK_BYTES && b >= t.s[i].src && b < t.s[i].src + t.s[i].len) return t.s[i].off + (b - t.s[i].src);
    return ~0u;
}
constexpr int state_section_of_kind(const StateLayout &t, uint8_t kind) {
    for (int i = 0; i < STATE_SECTIONS; i++)
        if (t.s[i].kind == kind) return i;
    return -1;
}
static constexpr uint32_t STATE_OFF_LCDC = state_file_byte(STATE_LAYOUT, state_reg_byte(R_LCD0, 0));
static constexpr uint32_t STATE_OFF_STAT = state_file_byte(STATE_LAYOUT, state_reg_byte(R_LCD0, 1));
static constexpr uint32_t STATE_OFF_CGB = state_file_byte(STATE_LAYOUT, state_reg_byte(R_HDR, 3));
static constexpr int STATE_FB_SECTION = state_section_of_kind(STATE_LAYOUT, SK_FB);
static_assert(STATE_OFF_CGB == 4 && STATE_OFF_LCDC == 8375 && STATE_LAYOUT.s[STATE_FB_SECTION].off == 9125, "v9 offsets (SURVEY.md 8c)");

__host__ __device__ inline int state_ctz64(uint64_t m) {
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)m) - 1;
#else
    return __builtin_ctzll(m);
#endif
}

// a screen word is one of PyBoy's four DMG values (SHADE_WORDS); the shade of one that is
__host__ __device__ inline bool state_shade_ok(uint32_t v) {
    return v == state_shade_word(0) || v == state_shade_word(1) || v == state_shade_word(2) || v == state_shade_word(3);
}
__host__ __device__ inline uint32_t state_shade_of(uint32_t v) {
    return v == state_shade_word(1) ? 1u : v == state_shade_word(2) ? 2u : v == state_shade_word(3) ? 3u : 0u;
}

// Image word j of the canonical image of a v9 file.  `secs` has bit s set for the sections that may give word j bits (a
// superset is fine: the others give none); rd(o) returns file bytes o .. o + 3 as a little-endian word, of which only the
// bytes inside those sections are used.  Per section kind, the inverse of state_byte: SK_BYTES bytes go back into their
// word, an SK_FIELD byte is masked and shifted into place, a scanline record is its 4 bytes plus 0x10 when byte 4 is
// non-zero (blob_to_image's rule, not bit 0 shifted), and 16 screen words become 16 two-bit shades.  Where two sections
// give the same bits (the second copies of double_speed and cgb) the first in file order wins; the bits no section gives
// are state_unfiled_bits.  For a file state_row_valid accepts this is blob_to_image's word.
template <class Rd>
__host__ __device__ inline uint32_t state_image_word(const StateLayout &t, uint64_t secs, uint32_t j, const Rd &rd) {
    uint32_t w = 0, have = 0;
    for (; secs; secs &= secs - 1) {
        const StateSection &s = t.s[state_ctz64(secs)];
        uint32_t v = 0, m = ~0u;
        if (s.kind == SK_BYTES) {
            const uint32_t b0 = 4 * j > s.src ? 4 * j : s.src, b1 = 4 * j + 4 < s.src + s.len ? 4 * j + 4 : s.src + s.len;
            if (b0 >= b1) continue;
            m = (0xFFFFFFFFu >> (32 - 8 * (b1 - b0))) << (8 * (b0 & 3));
            v = rd(s.off + (b0 - s.src)) << (8 * (b0 & 3));
        } else if (s.kind == SK_FIELD) {
            if (j != s.src) continue;
            m = (uint32_t)s.mask << s.shift;
            v = rd(s.off) << s.shift;
        } else if (s.kind == SK_LP) {
            const uint32_t r = j - IMG_LP;
            if (r >= LP_WORDS) continue;
            v = r & 1 ? (rd(s.off + 5 * (r >> 1) + 4) & 0xFF ? 0x10u : 0u) : rd(s.off + 5 * (r >> 1));
        } else if (s.kind == SK_FB) {
            const uint32_t q = j - IMG_FB;
            if (q >= FB_WORDS) continue;
            for (uint32_t p = 0; p < 16; p++) v |= state_shade_of(rd(s.off + 64 * q + 4 * p)) << (2 * p);
        } else {
            continue;
        }
        w |= v & m & ~have;
        have |= m;
    }
    return w | state_unfiled_bits(j, j == IMG_REGS + R_LCD2 ? rd(STATE_OFF_STAT) : 0u);
}

// blob_to_image's acceptance rules for a v9 file (whose length is fixed): every SK_CONST section holds its constant (the
// version byte is 9, the high halves of clock and clock_target are 0), the cgb byte is 0, and every screen word is one of
// PyBoy's four DMG values.  state_head_ok is all but the screen; rd(o) as for state_image_word.
template <class Rd>
__host__ __device__ inline bool state_head_ok(const StateLayout &t, const Rd &rd) {
    bool ok = (rd(STATE_OFF_CGB) & 0xFF) == 0;
    for (int i = 0; i < STATE_SECTIONS; i++)
        if (t.s[i].kind == SK_CONST)
            for (uint32_t o = t.s[i].off; o < t.s[i].off + t.s[i].len; o++) ok &= (rd(o) & 0xFF) == t.s[i].src;
    return ok;
}
template <class Rd>
__host__ __device__ inline bool state_row_valid(const StateLayout &t, const Rd &rd) {
    bool ok = state_head_ok(t, rd);
    const StateSection &fb = t.s[STATE_FB_SECTION];
    for (uint32_t o = fb.off; o < fb.off + fb.len; o += 4) ok &= state_shade_ok(rd(o));
    return ok;
}

// PyBoy v9 / v7 blob -> canonical image (layout: SURVEY.md 8c).  Returns 0 or a negative error.
static int blob_to_image(const uint8_t *b, size_t len, std::vector<uint32_t> &img, int *version_out, std::string &err) {
    if (len < 1) { err = "empty save-state"; return GBENV_E_STATE; }
    int ver = b[0];
    if (!((ver == 9 && len == 142610) || (ver == 7 && len == 142586))) {
        err = "unsupported PyBoy save-state (need v9/142610 B or v7/142586 B)";
        return GBENV_E_STATE;
    }
    img.assign(IMG_WORDS, 0);
    const uint8_t *p = b + 1;
    uint32_t hdr = *p++;  // bootrom_enabled
    if (ver >= 8) {
        hdr |= (uint32_t)p[0] << 8 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 24;
        if (p[2]) { err = "CGB save-states are not supported"; return GBENV_E_STATE; }
        p += 3;
    }
    uint32_t A = p[0], F = p[1], B = p[2], C = p[3], D = p[4], E = p[5];
    uint32_t HL = p[6] | (p[7] << 8), SP = p[8] | (p[9] << 8), PC = p[10] | (p[11] << 8);
    uint32_t ime = p[12], halted = p[13], stopped = p[14], IE = p[15], iq = 0, IF = 0;
    p += 16;
    if (ver >= 8) { iq = p[0]; IF = p[1]; p += 2; }
    uint32_t *regs = &img[IMG_REGS];
    regs[R_BCDE] = C | (B << 8) | (E << 16) | (D << 24);
    regs[R_HLAF] = HL | (A << 16) | (F << 24);
    regs[R_SPPC] = SP | (PC << 16);
    regs[R_INT] = (ime & 1) | ((halted & 1) << 1) | ((stopped & 1) << 2) | ((iq & 1) << 3) | (IE << 8) | (IF << 16);
    for (uint32_t i = 0; i < 0x2000; i++) img_set_byte(img, IMG_MEM, MEM_VRAM + i, *p++);
    for (uint32_t i = 0; i < 0xA0; i++) img_set_byte(img, IMG_MEM, MEM_HI + i, *p++);
    uint32_t LCDC = p[0], BGP = p[1], OBP0 = p[2], OBP1 = p[3], STAT = p[4], LY = p[5], LYC = p[6], SCY = p[7], SCX = p[8], WY = p[9], WX = p[10];
    p += 11;
    uint64_t clock = 0, target = 0;
    uint32_t next_mode = 2;
    if (ver >= 8) {
        p += 2;
        for (int i = 7; i >= 0; i--) clock = (clock << 8) | p[i];
        p += 8;
        for (int i = 7; i >= 0; i--) target = (target << 8) | p[i];
        p += 8;
        next_mode = *p++;
        if (clock > 0xFFFFFFFFull || target > 0xFFFFFFFFull) { err = "LCD clock out of range"; return GBENV_E_STATE; }
    }
    regs[R_LCD0] = LCDC | (STAT << 8) | (LY << 16) | (LYC << 24);
    regs[R_LCD1] = SCY | (SCX << 8) | (WY << 16) | (WX << 24);
    regs[R_LCD2] = BGP | (OBP0 << 8) | (OBP1 << 16) | ((next_mode & 3) << 26) | state_unfiled_bits(IMG_REGS + R_LCD2, STAT);
    regs[R_CLOCK] = (uint32_t)clock;
    regs[R_TARGET] = (uint32_t)target;
    for (uint32_t y = 0; y < 144; y++, p += 5) {
        img[IMG_LP + 2 * y] = p[0] | (p[1] << 8) | (p[2] << 16) | (p[3] << 24);  // SCX SCY WX(raw) WY
        img[IMG_LP + 2 * y + 1] = p[4] ? 0x10u : 0u;                              // tile_data_select
    }
    for (uint32_t i = 0; i < 144 * 160; i++, p += 4) {
        uint32_t wv = p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24);
        int shade = -1;
        for (int s = 0; s < 4; s++)
            if (wv == SHADE_WORDS[s]) shade = s;
        if (shade < 0 && wv == 0) shade = 3;
        if (shade < 0) { err = "framebuffer word is not one of PyBoy's four DMG values"; return GBENV_E_STATE; }
        img[IMG_FB + (i >> 4)] |= (uint32_t)shade << (2 * (i & 15));
    }
    for (uint32_t i = 0; i < 0x2000; i++) img_set_byte(img, IMG_MEM, MEM_WRAM + i, *p++);
    for (uint32_t i = 0; i < 96; i++) img_set_byte(img, IMG_MEM, MEM_HI + 0xA0 + i, *p++);
    for (uint32_t i = 0; i < 76; i++) img_set_byte(img, IMG_MEM, MEM_HI + 0x100 + i, *p++);
    for (uint32_t i = 0; i < 127; i++) img_set_byte(img, IMG_MEM, MEM_HI + 0x180 + i, *p++);
    for (uint32_t i = 0; i < 52; i++) img_set_byte(img, IMG_MEM, MEM_HI + 0x14C + i, *p++);
    uint32_t DIV = p[0], TIMA = p[1], DIVC = p[2] | (p[3] << 8), TIMAC = p[4] | (p[5] << 8), TMA = p[6], TAC = p[7];
    p += 8;
    regs[R_TIMER] = DIV | (TIMA << 8) | (TMA << 16) | (TAC << 24);
    regs[R_DIVC] = DIVC;
    regs[R_TIMAC] = TIMAC;
    regs[R_MBC] = p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24);
    p += 4;
    for (uint32_t i = 0; i < 0x8000; i++) img_set_byte(img, IMG_CRAM, i, *p++);
    regs[R_JOY] = p[0] | (p[1] << 8) | state_unfiled_bits(IMG_REGS + R_JOY, 0);  // ly_window kept by the merge, lp_dirty = 144
    p += 2;
    regs[R_HDR] = hdr;
    regs[R_MISC] = state_unfiled_bits(IMG_REGS + R_MISC, 0);
    if ((size_t)(p - b) != len) { err = "save-state length mismatch"; return GBENV_E_STATE; }
    *version_out = ver;
    return GBENV_OK;
}

static inline void image_to_blob(const std::vector<uint32_t> &img, uint8_t *b) {
    for (const StateSection &s : STATE_LAYOUT.s)
        for (uint32_t o = s.off; o < s.off + s.len; o++) b[o] = state_byte(s, o, s.kind == SK_CONST ? 0u : img[state_word(s, o)]);
}

// fresh post-boot DMG machine (our convention; mirrors oracle gb_power_on)
static void power_on_image(std::vector<uint32_t> &img) {
    img.assign(IMG_WORDS, 0);
    uint32_t *regs = &img[IMG_REGS];
    regs[R_BCDE] = 0x13 | (0x00 << 8) | (0xD8 << 16) | (0x00u << 24);
    regs[R_HLAF] = 0x014D | (0x01 << 16) | (0xB0u << 24);
    regs[R_SPPC] = 0xFFFE | (0x0100u << 16);
    regs[R_INT] = 0;
    regs[R_LCD0] = 0x91 | (0x80 << 8);
    regs[R_LCD1] = 0;
    regs[R_LCD2] = 0xFC | (0xFF << 8) | (0xFF << 16) | ((0u | (2u << 2)) << 24);
    regs[R_MBC] = 1;
    regs[R_JOY] = 0x0F | (0x0F << 8) | (0xFFu << 16) | (144u << 24);
    regs[R_MISC] = 0xFF;
    img_set_byte(img, IMG_MEM, MEM_HI + 0x100, 0xFF);      // P1
    img_set_byte(img, IMG_MEM, MEM_HI + 0x14C + 4, 0x01);  // FF50
    for (uint32_t i = 0; i < FB_WORDS; i++) img[IMG_FB + i] = 0xFFFFFFFFu;  // PyBoy's fresh screen buffer is all zero words = black
    for (uint32_t y = 0; y < 144; y++) img[IMG_LP + 2 * y] = 7u << 16;      // fresh _scanlineparameters hold WX - 7 = 0
}

