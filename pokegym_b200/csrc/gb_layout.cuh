// gb_layout.cuh -- HBM layout of the batched Game Boy state (see DESIGN.md "Data layout").
//
// Envs are grouped in tiles of 32 (= one warp in the emulation kernel, lane == env % 32).  Every
// per-env array is stored word-interleaved ("SoA, address-major / env-minor at 4-byte granule"):
//     word w of env (tile t, lane l)  ->  base[(t * WORDS + w) * 32 + l]        (uint32_t units)
// so when the 32 envs of a warp touch the same Game Boy address -- the common case, they run the same
// ROM -- the warp reads or writes one fully used 128-byte line, and a 16-bit stack push/pop or a
// sequential copy inside one env stays inside one 32-byte sector.
#pragma once
#include <stdint.h>
#include "gb_hd.h"

#define GB_TILE 32

#define FRAME_CYCLES 70224u

// --- plain-RAM array "mem": VRAM | WRAM | HI page (0xFE00-0xFFFF)
#define MEM_VRAM 0x0000u  // 0x8000-0x9FFF
#define MEM_WRAM 0x2000u  // 0xC000-0xDFFF (echo 0xE000-0xFDFF redirects here)
#define MEM_HI 0x4000u    // 0xFE00-0xFFFF: OAM, 0xFEA0-FEFF, IO array, 0xFF4C-7F, HRAM
#define MEM_BYTES 0x4200u
#define MEM_WORDS (MEM_BYTES / 4)

#define CRAM_BYTES 0x8000u  // 4 x 8 KiB MBC3 RAM banks
#define CRAM_WORDS (CRAM_BYTES / 4)

// --- framebuffer: 2 bits per pixel (shade after palette), 16 pixels per word, 10 words per line.
// PyBoy's 32-bit framebuffer words only take four values and the low "colour-0" flag byte is 1
// exactly when the shade is white (oracle/gb_core.h GBQ_COL0_FLAG_FOLLOWS_SHADE), so 2 bpp is lossless.
#define FB_LINE_WORDS 10
#define FB_WORDS (144 * FB_LINE_WORDS)

// --- per-scanline renderer parameters (PyBoy Renderer._scanlineparameters), 2 words per line
//     word0 = SCX | SCY<<8 | WX<<16 | WY<<24     word1 = LCDC (tile_data_select = bit 4)
#define LP_WORDS (144 * 2)

// --- deferred-line records (gb_device.cuh "deferred PPU"): what Renderer.scanline needs besides VRAM / OAM, captured at the
//     HBlank of each visible line of the frame that is rendered: word0 = SCX | SCY<<8 | WX<<16 | WY<<24, word1 = LCDC | BGP<<8 |
//     OBP0<<16 | OBP1<<24, word2 = Renderer.ly_window before the line.  Scratch between k_run_frames and k_render_pending,
//     not part of the env's state image.
#define DL_WORDS (144 * 3)

// --- CPU / LCD / timer / MBC / joypad registers, one word each (see struct Regs in gb_device.cuh)
enum {
    R_BCDE = 0,   // C | B<<8 | E<<16 | D<<24
    R_HLAF,       // L | H<<8 | A<<16 | F<<24
    R_SPPC,       // SP | PC<<16
    R_INT,        // ime | halted<<1 | stopped<<2 | interrupt_queued<<3 | fault<<4 | IE<<8 | IF<<16
    R_LCD0,       // LCDC | STAT<<8 | LY<<16 | LYC<<24
    R_LCD1,       // SCY | SCX<<8 | WY<<16 | WX<<24
    R_LCD2,       // BGP | OBP0<<8 | OBP1<<16 | (stat_mode | next_stat_mode<<2 | disable_renderer<<4 | frame_done<<5)<<24
    R_CLOCK,      // lcd.clock
    R_TARGET,     // lcd.clock_target
    R_TIMER,      // DIV | TIMA<<8 | TMA<<16 | TAC<<24
    R_DIVC,       // timer.DIV_counter
    R_TIMAC,      // timer.TIMA_counter
    R_MBC,        // rombank | rambank<<8 | ram_enabled<<16 | memorymodel<<24
    R_JOY,        // directional | standard<<8 | (ly_window & 0xFF)<<16 | lp_dirty<<24
    R_HDR,        // bootrom_enabled | key1<<8 | double_speed<<16 | cgb<<24
    R_MISC,       // blank_shade (0..3, 0xFF = framebuffer not uniformly blank) | defer_from<<8 | defer_next<<16 (lines awaiting k_render_pending)
    R_WORDS
};

// --- visited bitmaps (seen_coords / screen_memory, gb_wrap.cuh WrapArrays): per env a page table of WRAP_MAPS maps x
//     VIS_BANDS row bands, each entry a page index + 1 (0 = no page); a page holds 64 rows x 256 columns, bit x & 31 of word
//     x / 32 of a row being column x.  Shared with the packed-observation writer (gb_obs.cu).
#define WRAP_MAPS 248
#define VIS_ROW_WORDS 8                       // 256 columns / 32
#define VIS_BAND_ROWS 64                      // a visited-bitmap page covers 64 rows x 256 columns of one map = 2 KiB
#define VIS_BANDS 4
#define VIS_PAGE_WORDS (VIS_BAND_ROWS * VIS_ROW_WORDS)
#define VIS_PT_ENTRIES (WRAP_MAPS * VIS_BANDS)  // page-table entries per env

// canonical linear per-env image used by templates / save_state staging (uint32_t words)
#define IMG_MEM 0
#define IMG_CRAM (IMG_MEM + MEM_WORDS)
#define IMG_FB (IMG_CRAM + CRAM_WORDS)
#define IMG_LP (IMG_FB + FB_WORDS)
#define IMG_REGS (IMG_LP + LP_WORDS)
#define IMG_WORDS (IMG_REGS + R_WORDS)

struct DevArrays {
    uint32_t *mem;   // [tiles][MEM_WORDS][32]
    uint32_t *cram;  // [tiles][CRAM_WORDS][32]
    uint32_t *fb;    // [tiles][FB_WORDS][32]
    uint32_t *lp;    // [tiles][LP_WORDS][32]
    uint32_t *regs;  // [tiles][R_WORDS][32]
    uint32_t *dl;    // [tiles][DL_WORDS][32]; may be null (no deferred rendering)
    const uint8_t *rom;
    const uint4 *rom_dec;  // pre-decoded ROM: one 16-byte control word per ROM offset (gb_predecode.h)
    uint32_t rom_banks;
    int n_envs;
    int n_tiles;
};

__host__ __device__ inline size_t il_index(int tile, uint32_t words_per_env, uint32_t w, int lane) {
    return ((size_t)tile * words_per_env + w) * GB_TILE + (size_t)lane;
}
// scanline parameters are interleaved as 8-byte pairs so one line is a single 64-bit store
__host__ __device__ inline size_t lp_index(int tile, uint32_t w, int lane) {
    return (size_t)tile * LP_WORDS * GB_TILE + ((size_t)(w >> 1) * GB_TILE + (size_t)lane) * 2 + (w & 1);
}

// Canonical per-env image <-> interleaved arrays.  image word j of env e lives at:
//   IMG_MEM..: mem, IMG_CRAM..: cram, IMG_FB..: fb, IMG_LP..: lp (pair-interleaved), IMG_REGS..: regs
__device__ __forceinline__ uint32_t *image_slot(const DevArrays &d, int env, uint32_t j) {
    int tile = env >> 5, lane = env & 31;
    if (j < IMG_CRAM) return d.mem + il_index(tile, MEM_WORDS, j - IMG_MEM, lane);
    if (j < IMG_FB) return d.cram + il_index(tile, CRAM_WORDS, j - IMG_CRAM, lane);
    if (j < IMG_LP) return d.fb + il_index(tile, FB_WORDS, j - IMG_FB, lane);
    if (j < IMG_REGS) return d.lp + lp_index(tile, j - IMG_LP, lane);
    return d.regs + il_index(tile, R_WORDS, j - IMG_REGS, lane);
}

// PyBoy load_state semantics that depend on the env's previous state (oracle GBQ_STAT_LOAD_KEEPS_MODE):
// STAT bits 0-2 and STATRegister._mode survive a load; LCD-off states force mode 0 through set_lcdc.
// For v7 blobs clock / clock_target / next_stat_mode / IF / interrupt_queued are not in the file.
__device__ __forceinline__ uint32_t merge_loaded_reg(uint32_t r, uint32_t old, uint32_t neu, int version, uint32_t new_lcdc) {
    if (version == 0) return neu;  // raw image (power-on): no PyBoy load_state semantics
    bool lcd_off = !(new_lcdc & 0x80);
    if (r == R_LCD0) {
        uint32_t old_stat = (old >> 8) & 0xFF;
        if (lcd_off) old_stat &= 0xFC;  // set_lcdc -> STAT.set_mode(0)
        uint32_t stat = (old_stat & 0x87) | ((neu >> 8) & 0x78);
        return (neu & 0xFFFF00FFu) | (stat << 8);
    }
    if (r == R_LCD2) {
        uint32_t oldf = old >> 24, mode = oldf & 3, next = (neu >> 26) & 3;
        if (lcd_off) mode = 0;
        if (version < 8) next = lcd_off ? 2 : ((oldf >> 2) & 3);
        return (neu & 0x00FFFFFFu) | ((mode | (next << 2) | (oldf & 0x30)) << 24);
    }
    if (r == R_JOY) return (neu & 0xFF00FFFFu) | (old & 0x00FF0000u);  // Renderer.ly_window is not serialised
    if (version < 8) {
        if (r == R_CLOCK) return lcd_off ? 0 : old;
        if (r == R_TARGET) return lcd_off ? FRAME_CYCLES : old;
        if (r == R_INT) return (neu & 0x0000FF17u) | (old & 0x00FF0008u);  // keep IF and interrupt_queued
    }
    return neu;
}
