// gb_device.cuh -- device-side Game Boy (DMG + MBC3) machine: SM83 interpreter, bus, timer, LCD
// state machine and scanline renderer, one env per thread.
//
// Replaces PyBoy 1.6.x as driven by /root/reference/pokegym/pyboy_binding.py:71-91 (24 x PyBoy.tick
// per env step) and every get/set_memory_value call of the reference wrapper.  Semantics follow the
// instruction-granular PyBoy model of SURVEY.md Appendix A (peripherals advance after each whole
// instruction, interrupt dispatch costs 0 cycles, HALT fast-forwards to the next LCD event, one
// TIMA increment and one LCD mode change per tick at most ...).  Structure is B200-first and shares
// nothing with the CPU oracle: registers are packed words decoded with bit-field arithmetic, all
// env state lives in word-interleaved HBM arrays (gb_layout.cuh), and the main loop is organised
// around LCD events so the 32 envs of a warp re-converge at every scanline boundary.
#pragma once
#include "gb_hd.h"
#include "gb_layout.cuh"

#define FLAG_Z 0x80u
#define FLAG_N 0x40u
#define FLAG_H 0x20u
#define FLAG_C 0x10u

#define IRQ_VBLANK 0x01u
#define IRQ_STAT 0x02u
#define IRQ_TIMER 0x04u
#define IRQ_SERIAL 0x08u
#define IRQ_JOYPAD 0x10u

#define M_SCX(m) ((m).scroll & 0xFF)
#define M_SCY(m) (((m).scroll >> 8) & 0xFF)
#define M_WX(m) (((m).scroll >> 16) & 0xFF)
#define M_WY(m) ((m).scroll >> 24)
#define M_BGP(m) ((m).pal & 0xFF)
#define M_OBP0(m) (((m).pal >> 8) & 0xFF)
#define M_OBP1(m) (((m).pal >> 16) & 0xFF)
#define M_TIMA(m) (((m).tmr >> 8) & 0xFF)
#define M_TMA(m) (((m).tmr >> 16) & 0xFF)
#define M_TAC(m) ((m).tmr >> 24)

struct Machine {
    // SM83 registers: C|B<<8|E<<16|D<<24 and L|H<<8|A<<16|F<<24 (pairs are native little-endian halves)
    uint32_t bcde, hlaf, sp, pc;
    uint32_t ime, halted, stopped, iq, fault, ie, iflag;
    // LCD
    // hot LCD registers unpacked; the rest stay packed the way the out-of-line IO / renderer paths consume them
    uint32_t lcdc, stat, ly, lyc;
    uint32_t scroll;  // SCX | SCY<<8 | WX<<16 | WY<<24  (the order of PyBoy's per-scanline parameter record)
    uint32_t pal;     // BGP | OBP0<<8 | OBP1<<16
    uint32_t stat_mode, next_mode, disable_renderer, frame_done;
    uint32_t clock, target;
    // timer
    uint32_t div, divc, timac;
    uint32_t tmr;  // TIMA<<8 | TMA<<16 | TAC<<24
    // MBC3
    uint32_t rombank, rambank, ram_en, memorymodel, rom_off;
    // joypad + renderer bookkeeping
    uint32_t joy_dir, joy_std, lp_dirty, blank_shade;
    int ly_window;
    uint32_t hdr;
    // statistics (n_cycles = clock delta + cyc_adj, see machine_store)
    uint32_t n_instr, n_cycles, cyc_adj, clock0;
    uint32_t lazy;  // k_run_frames: soft LCD events may be applied late (set by lcd_deadline)
    // deferred PPU: lines [defer_from, defer_next) of the rendered frame are recorded in `dl` and not yet drawn; defer_active:
    // a line of the current frame has been recorded (from then on VRAM / OAM writes leave the fast loop and flush first)
    uint32_t defer_from, defer_next, defer_active;
    uint32_t *dl;  // this env's deferred-line records (word k of line y at dl[(y * 3 + k) * 32]), or null: render at once
    int t_sync;  // k_run_frames: value of the interpreter's cycle countdown when clock / divc were last brought up to date
    // memory (pointers already offset to this env's lane inside its tile)
    uint8_t *memb;   // plain RAM, byte i at memb[((i >> 2) << 7) | (i & 3)]
    uint8_t *cramb;  // cart RAM, same addressing
    uint32_t *fb;    // word w at fb[w * 32]
    uint2 *lp;       // scanline y at lp[y * 32]
    const uint8_t *rom;
    uint32_t rom_banks;
    // k_run_frames: this env's renderer scratch in shared memory (10-word line buffer and 10 sprite sort keys, stride rls)
    uint32_t rls;
    uint32_t *rline, *rkeys;
};

// ------------------------------------------------------------------------------- state load/store

__device__ __forceinline__ void machine_bind(Machine &m, const DevArrays &d, int tile, int lane) {
    m.memb = (uint8_t *)(d.mem + il_index(tile, MEM_WORDS, 0, lane));
    m.cramb = (uint8_t *)(d.cram + il_index(tile, CRAM_WORDS, 0, lane));
    m.fb = d.fb + il_index(tile, FB_WORDS, 0, lane);
    m.lp = (uint2 *)(d.lp + (size_t)tile * LP_WORDS * GB_TILE) + lane;
    m.rom = d.rom;
    m.rom_banks = d.rom_banks;
    m.dl = nullptr;  // the emulation kernel switches deferred rendering on (RunParams.defer)
}

__device__ __forceinline__ void machine_set_rombank(Machine &m, uint32_t bank) {
    m.rombank = bank;
    m.rom_off = (bank % m.rom_banks) * 0x4000u - 0x4000u;  // rom[addr + rom_off] for 0x4000 <= addr < 0x8000
}

__device__ inline void machine_load(Machine &m, const DevArrays &d, int tile, int lane) {
    machine_bind(m, d, tile, lane);
    const uint32_t *r = d.regs + il_index(tile, R_WORDS, 0, lane);
    uint32_t w;
    m.bcde = r[R_BCDE * 32];
    m.hlaf = r[R_HLAF * 32];
    w = r[R_SPPC * 32];
    m.sp = w & 0xFFFF;
    m.pc = w >> 16;
    w = r[R_INT * 32];
    m.ime = w & 1; m.halted = (w >> 1) & 1; m.stopped = (w >> 2) & 1; m.iq = (w >> 3) & 1; m.fault = (w >> 4) & 1;
    m.ie = (w >> 8) & 0xFF; m.iflag = (w >> 16) & 0xFF;
    w = r[R_LCD0 * 32];
    m.lcdc = w & 0xFF; m.stat = (w >> 8) & 0xFF; m.ly = (w >> 16) & 0xFF; m.lyc = w >> 24;
    w = r[R_LCD1 * 32];
    m.scroll = ((w & 0x00FF00FFu) << 8) | ((w >> 8) & 0x00FF00FFu);  // R_LCD1 holds SCY SCX WY WX
    w = r[R_LCD2 * 32];
    m.pal = w & 0xFFFFFFu;
    m.stat_mode = (w >> 24) & 3; m.next_mode = (w >> 26) & 3; m.disable_renderer = (w >> 28) & 1; m.frame_done = (w >> 29) & 1;
    m.clock = r[R_CLOCK * 32];
    m.target = r[R_TARGET * 32];
    w = r[R_TIMER * 32];
    m.div = w & 0xFF; m.tmr = w & 0xFFFFFF00u;
    m.divc = r[R_DIVC * 32];
    m.timac = r[R_TIMAC * 32];
    w = r[R_MBC * 32];
    m.rambank = (w >> 8) & 0xFF; m.ram_en = (w >> 16) & 0xFF; m.memorymodel = w >> 24;
    machine_set_rombank(m, w & 0xFF);
    w = r[R_JOY * 32];
    m.joy_dir = w & 0xFF; m.joy_std = (w >> 8) & 0xFF; m.ly_window = (int)(int8_t)((w >> 16) & 0xFF); m.lp_dirty = w >> 24;
    m.hdr = r[R_HDR * 32];
    w = r[R_MISC * 32];
    m.blank_shade = w & 0xFF;
    m.defer_from = m.defer_next = m.defer_active = 0;  // what the last launch left pending (bits 8-23) has been drawn by k_render_pending
    m.n_instr = 0;
    m.n_cycles = 0;
    m.cyc_adj = 0;
    m.clock0 = m.clock;
    m.t_sync = 0;
    m.lazy = 0;
}

__device__ inline void machine_store(Machine &m, const DevArrays &d, int tile, int lane) {
    uint32_t *r = d.regs + il_index(tile, R_WORDS, 0, lane);
    m.div = (m.div + (m.divc >> 8)) & 0xFF;  // DIV is kept lazily: fold the accumulated cycles (Timer.tick is additive)
    m.divc &= 0xFF;
    m.n_cycles = m.clock - m.clock0 + m.cyc_adj;
    r[R_BCDE * 32] = m.bcde;
    r[R_HLAF * 32] = m.hlaf;
    r[R_SPPC * 32] = (m.sp & 0xFFFF) | (m.pc << 16);
    r[R_INT * 32] = m.ime | (m.halted << 1) | (m.stopped << 2) | (m.iq << 3) | (m.fault << 4) | (m.ie << 8) | (m.iflag << 16);
    r[R_LCD0 * 32] = m.lcdc | (m.stat << 8) | (m.ly << 16) | (m.lyc << 24);
    r[R_LCD1 * 32] = ((m.scroll & 0x00FF00FFu) << 8) | ((m.scroll >> 8) & 0x00FF00FFu);
    r[R_LCD2 * 32] = m.pal | ((m.stat_mode | (m.next_mode << 2) | (m.disable_renderer << 4) | (m.frame_done << 5)) << 24);
    r[R_CLOCK * 32] = m.clock;
    r[R_TARGET * 32] = m.target;
    r[R_TIMER * 32] = m.div | m.tmr;
    r[R_DIVC * 32] = m.divc;
    r[R_TIMAC * 32] = m.timac;
    r[R_MBC * 32] = m.rombank | (m.rambank << 8) | (m.ram_en << 16) | (m.memorymodel << 24);
    r[R_JOY * 32] = m.joy_dir | (m.joy_std << 8) | (((uint32_t)m.ly_window & 0xFF) << 16) | (m.lp_dirty << 24);
    r[R_HDR * 32] = m.hdr;
    r[R_MISC * 32] = m.blank_shade | (m.defer_from << 8) | (m.defer_next << 16);
}

// ----------------------------------------------------------------------------------- plain memory

__device__ __forceinline__ uint32_t mem_rd(const Machine &m, uint32_t i) { return m.memb[((i >> 2) << 7) | (i & 3)]; }
__device__ __forceinline__ void mem_wr(Machine &m, uint32_t i, uint32_t v) { m.memb[((i >> 2) << 7) | (i & 3)] = (uint8_t)v; }
__device__ __forceinline__ uint32_t mem_rd_word(const Machine &m, uint32_t w) { return ((const uint32_t *)m.memb)[w << 5]; }
__device__ __forceinline__ void mem_wr_word(Machine &m, uint32_t w, uint32_t v) { ((uint32_t *)m.memb)[w << 5] = v; }
__device__ __forceinline__ uint32_t vram_rd16(const Machine &m, uint32_t i) {  // i even: both bytes share a word
    return *(const uint16_t *)(m.memb + (((i >> 2) << 7) | (i & 2)));
}

// ------------------------------------------------------------------------------------------ joypad

__device__ __forceinline__ uint32_t joypad_pull(const Machine &m, uint32_t v) {  // Interaction.pull
    uint32_t p14 = (v >> 4) & 1, p15 = (v >> 5) & 1, b = (v | 0xCF) & 0xFF;
    if (p14 != p15) b &= p14 ? m.joy_std : m.joy_dir;  // only one group selected: byte &= 4-bit nibble
    return b;
}

__device__ __forceinline__ void joypad_event(Machine &m, int button, int pressed) {  // Interaction.key_event
    uint32_t bit = 1u << (button & 3);
    uint32_t &reg = (button < 4) ? m.joy_dir : m.joy_std;
    uint32_t before = reg;
    reg = pressed ? (reg & ~bit) : (reg | bit);
    if ((before ^ reg) & before) m.iflag |= IRQ_JOYPAD;
}

// --------------------------------------------------------------------------------------------- LCD

__device__ __forceinline__ uint32_t stat_set_mode(Machine &m, uint32_t mode) {
    if (m.stat_mode == mode) return 0;
    m.stat_mode = mode;
    m.stat = (m.stat & 0xFC) | mode;
    return (mode != 3 && ((m.stat >> (mode + 3)) & 1)) ? IRQ_STAT : 0;
}

__device__ __forceinline__ uint32_t stat_update_lyc(Machine &m) {
    if (m.lyc == m.ly) {
        m.stat |= 0x04;
        return (m.stat & 0x40) ? IRQ_STAT : 0;
    }
    m.stat &= 0xFB;
    return 0;
}

__device__ __forceinline__ void lcd_set_lcdc(Machine &m, uint32_t v) {
    if ((v ^ m.lcdc) & 0x10) m.lp_dirty = 144;
    m.lcdc = v;
    if (!(v & 0x80)) {
        m.cyc_adj += m.clock;
        m.clock = 0;
        m.target = FRAME_CYCLES;
        stat_set_mode(m, 0);
        m.next_mode = 2;
        m.ly = 0;
        m.lp_dirty = 144;  // line order restarts after an LCD-off period
    }
}

// 2-bit shade for colour index idx through palette register pal
__device__ __forceinline__ uint32_t pal_shade(uint32_t pal, uint32_t idx) { return (pal >> (idx * 2)) & 3; }

// One tile row (rowdata = plane 0 | plane 1 << 8, leftmost pixel = bit 7 of each plane) -> 8 pixels x 2-bit colour
// index, leftmost pixel at bit 0.  Both planes are bit-reversed with one BREV, moved to the two half-words with one
// PRMT and spread to even bit positions together; `xflip` (sprites) skips the reversal.
__device__ __forceinline__ uint32_t tile_row_indices(uint32_t rowdata, bool xflip = false) {
    uint32_t x = xflip ? __byte_perm(rowdata, 0, 0x4140) : __byte_perm(__brev(rowdata), 0, 0x4243);  // plane0 | plane1 << 16
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return (x | (x >> 15)) & 0xFFFFu;
}

// map packed 2-bit colour indices (8 in a half-word or 16 in a word) through a palette register -> packed 2-bit shades
__device__ __forceinline__ uint32_t apply_palette(uint32_t idx, uint32_t pal) {
    uint32_t lo = idx & 0x55555555u, hi = (idx >> 1) & 0x55555555u;
    uint32_t m0 = ~lo & ~hi & 0x55555555u, m1 = lo & ~hi, m2 = ~lo & hi, m3 = lo & hi;  // one bit per pixel at even positions
    uint32_t s = 0;
    s |= m0 * (pal & 3);
    s |= m1 * ((pal >> 2) & 3);
    s |= m2 * ((pal >> 4) & 3);
    s |= m3 * ((pal >> 6) & 3);
    return s;
}

// RENDER_BATCH tiles of map row `row` (offset inside VRAM) from column `col` on (wrapping at 32), tile row `fine_y`:
// colour indices of their 8 pixels each.  All map bytes are loaded before the first tile row, all tile rows before the
// first use, so a batch costs two memory round trips; a batch may run past the last tile the caller needs (the
// addresses stay inside VRAM).
#define RENDER_BATCH 7
__device__ __forceinline__ void render_fetch_tiles(const Machine &m, uint32_t row, uint32_t col, uint32_t fine_y, uint32_t tds, uint32_t (&px)[RENDER_BATCH]) {
    uint32_t t[RENDER_BATCH];
#pragma unroll
    for (int j = 0; j < RENDER_BATCH; j++) t[j] = mem_rd(m, MEM_VRAM + row + ((col + j) & 31));
#pragma unroll
    for (int j = 0; j < RENDER_BATCH; j++) {
        const uint32_t tt = tds ? t[j] : (t[j] ^ 0x80) + 128;
        px[j] = vram_rd16(m, MEM_VRAM + tt * 16 + fine_y * 2);
    }
#pragma unroll
    for (int j = 0; j < RENDER_BATCH; j++) px[j] = tile_row_indices(px[j]);
}

// Renderer.scanline + Renderer.scanline_sprites for line y.  `line` is this thread's 10-word
// scratch in shared memory (stride `ls` words), `keys` its 10-entry sprite sort scratch.
__device__ inline void render_line(Machine &m, uint32_t y, uint32_t *line, uint32_t *keys, uint32_t ls) {
    const uint32_t lcdc = m.lcdc;
    const int wx = (int)M_WX(m) - 7, wy = (int)M_WY(m);
    const uint32_t scx = M_SCX(m), scy = M_SCY(m), bgp = M_BGP(m);
    const bool win_line = (lcdc & 0x20) && wy <= (int)y && wx < 160;
    if (win_line) m.ly_window += 1;
    const uint32_t tds = lcdc & 0x10;
    const int wstart = win_line ? (wx > 0 ? wx : 0) : 160;  // first screen x covered by the window

    // ---- background layer, x in [0, wstart)
    // Tiles are fetched seven at a time (render_fetch_tiles): seven independent map-byte loads, then seven independent
    // tile-row loads, so the two dependent VRAM accesses of a tile are paid once per batch, not once per tile.
    if (wstart > 0) {
        if (lcdc & 0x01) {
            const uint32_t map_base = (lcdc & 0x08) ? 0x1C00u : 0x1800u;
            const uint32_t row = map_base + ((((y + scy) >> 3) << 5) & 0x3FFu);
            const uint32_t fine_y = (y + scy) & 7;
            uint32_t col = scx >> 3;
            uint64_t acc = 0;
            int nbits = -(int)((scx & 7) * 2);  // drop the leftmost (scx & 7) pixels of the first tile
            uint32_t out = 0;
            const uint32_t nwords = ((uint32_t)wstart + 15) >> 4;
            while (out < nwords) {
                uint32_t px7[RENDER_BATCH];
                render_fetch_tiles(m, row, col, fine_y, tds, px7);
                col += RENDER_BATCH;
#pragma unroll
                for (int j = 0; j < RENDER_BATCH; j++) {
                    if (out < nwords) {
                        const uint32_t px = px7[j];
                        if (nbits < 0) acc = (uint64_t)(px >> (uint32_t)(-nbits));
                        else acc |= (uint64_t)px << nbits;
                        nbits += 16;
                        if (nbits >= 32) {
                            line[out * ls] = (uint32_t)acc;
                            out++;
                            acc >>= 32;
                            nbits -= 32;
                        }
                    }
                }
            }
        } else {
            for (uint32_t k = 0; k < ((uint32_t)wstart + 15) >> 4; k++) line[k * ls] = 0;  // colour 0 everywhere
        }
    }
    // ---- window layer, x in [wstart, 160)
    if (win_line) {
        const uint32_t map_base = (lcdc & 0x40) ? 0x1C00u : 0x1800u;
        const uint32_t lw = (uint32_t)m.ly_window;
        const uint32_t row = map_base + (((lw >> 3) << 5) & 0x3FFu);
        const uint32_t fine_y = lw & 7;
        uint32_t first = (uint32_t)(wstart - wx);  // window pixel index shown at x = wstart
        uint32_t col = first >> 3;
        uint32_t out = (uint32_t)wstart >> 4;
        uint32_t lead = ((uint32_t)wstart & 15) * 2;  // bits of word `out` that belong to the background
        uint64_t acc = lead ? (uint64_t)(line[out * ls] & ((1u << lead) - 1)) : 0;
        int nbits = (int)lead - (int)((first & 7) * 2);
        bool first_tile = true;
        while (out < FB_LINE_WORDS) {
            uint32_t px7[RENDER_BATCH];
            render_fetch_tiles(m, row, col, fine_y, tds, px7);
            col += RENDER_BATCH;
#pragma unroll
            for (int j = 0; j < RENDER_BATCH; j++) {
                if (out < FB_LINE_WORDS) {
                    uint32_t px = px7[j];
                    if (first_tile) {
                        px >>= (first & 7) * 2;
                        acc |= (uint64_t)px << lead;
                        nbits = (int)lead + 16 - (int)((first & 7) * 2);
                        first_tile = false;
                    } else {
                        acc |= (uint64_t)px << nbits;
                        nbits += 16;
                    }
                    if (nbits >= 32) {
                        line[out * ls] = (uint32_t)acc;
                        out++;
                        acc >>= 32;
                        nbits -= 32;
                    }
                }
            }
        }
    }
    if (y == 143) m.ly_window = -1;
    // ---- BG palette: colour indices -> shades, 16 pixels per word
#pragma unroll
    for (uint32_t k = 0; k < FB_LINE_WORDS; k++) line[k * ls] = apply_palette(line[k * ls], bgp);

    // ---- sprites
    if (lcdc & 0x02) {
        const int height = (lcdc & 0x04) ? 16 : 8;
        int count = 0;
        // pass 1: which of the 40 OAM entries overlap this line (independent loads, no early exit);
        // sy <= y < sy + height with sy = Y - 16  <=>  (unsigned)(y + 16 - Y) < height
        uint32_t hit_lo = 0, hit_hi = 0;
#pragma unroll
        for (uint32_t n = 0; n < 32; n++) hit_lo |= (uint32_t)((y + 16 - (mem_rd_word(m, (MEM_HI >> 2) + n) & 0xFF)) < (uint32_t)height) << n;
#pragma unroll
        for (uint32_t n = 0; n < 8; n++) hit_hi |= (uint32_t)((y + 16 - (mem_rd_word(m, (MEM_HI >> 2) + 32 + n) & 0xFF)) < (uint32_t)height) << n;
        // pass 2: the first ten in OAM order, sorted by (x, n)
        while ((hit_lo | hit_hi) && count < 10) {
            uint32_t n;
            if (hit_lo) { n = __ffs(hit_lo) - 1; hit_lo &= hit_lo - 1; }
            else { n = 32 + __ffs(hit_hi) - 1; hit_hi &= hit_hi - 1; }
            uint32_t e = mem_rd_word(m, (MEM_HI >> 2) + n);  // Y | X<<8 | tile<<16 | attr<<24
            {
                int sx = (int)((e >> 8) & 0xFF) - 8;
                // insertion into ascending (x, n) order; key = (sx + 8) << 8 | n keeps it unsigned
                uint32_t key = ((uint32_t)(sx + 8) << 8) | n;
                int j = count - 1;
                while (j >= 0 && keys[j * ls] > key) {
                    keys[(j + 1) * ls] = keys[j * ls];
                    j--;
                }
                keys[(j + 1) * ls] = key;
                count++;
            }
        }
        for (int i = count - 1; i >= 0; i--) {  // lowest priority first
            uint32_t n = keys[i * ls] & 0xFF;
            uint32_t e = mem_rd_word(m, (MEM_HI >> 2) + n);
            int sy = (int)(e & 0xFF) - 16, sx = (int)((e >> 8) & 0xFF) - 8;
            uint32_t tile = (e >> 16) & 0xFF, attr = e >> 24;
            if (height == 16) tile &= 0xFE;
            int dy = (int)y - sy;
            uint32_t yy = (attr & 0x40) ? (uint32_t)(height - dy - 1) : (uint32_t)dy;
            uint32_t rowdata = vram_rd16(m, MEM_VRAM + tile * 16 + yy * 2);
            uint32_t idx16 = tile_row_indices(rowdata, attr & 0x20);  // x flip: leftmost pixel = bit 0
            uint32_t opaque = (idx16 | (idx16 >> 1)) & 0x5555u;  // 1 per non-transparent pixel (even bit)
            uint32_t shades = apply_palette(idx16, (attr & 0x10) ? M_OBP1(m) : M_OBP0(m));
            // clip to the screen
            if (sx < 0) {
                uint32_t cut = (uint32_t)(-sx) * 2;
                opaque >>= cut;
                shades >>= cut;
                sx = 0;
            }
            if (sx >= 160 || opaque == 0) continue;
            uint32_t w = (uint32_t)sx >> 4, sh = ((uint32_t)sx & 15) * 2;
            uint64_t cur = line[w * ls];
            if (w + 1 < FB_LINE_WORDS) cur |= (uint64_t)line[(w + 1) * ls] << 32;
            uint64_t opq = (uint64_t)opaque << sh;
            if (w + 1 >= FB_LINE_WORDS) opq &= 0xFFFFFFFFull;  // pixels beyond x = 159
            if (attr & 0x80) {  // OBJ behind BG: only where the current pixel is white (flag == shade 0)
                uint64_t white = ~(cur | (cur >> 1)) & 0x5555555555555555ull;
                opq &= white;
            }
            uint64_t mask = opq | (opq << 1);
            cur = (cur & ~mask) | (((uint64_t)shades << sh) & mask);
            line[w * ls] = (uint32_t)cur;
            if (w + 1 < FB_LINE_WORDS) line[(w + 1) * ls] = (uint32_t)(cur >> 32);
        }
    }
    // ---- commit to the framebuffer (coalesced across the warp)
#pragma unroll
    for (uint32_t k = 0; k < FB_LINE_WORDS; k++) m.fb[(y * FB_LINE_WORDS + k) << 5] = line[k * ls];
    m.blank_shade = 0xFF;
}

// Out-of-line entry points of the renderer: inputs by value, so the caller's Machine stays in registers
// and the (large) renderer body is kept out of the interpreter's hot loop.
__device__ GB_NOINLINE int render_line_out(uint8_t *memb, uint32_t *fb, uint32_t lcdc, uint32_t scroll, uint32_t pal, int ly_window, uint32_t y,
                                            uint32_t *line, uint32_t *keys, uint32_t ls) {
    Machine r;
    r.memb = memb; r.fb = fb;
    r.lcdc = lcdc; r.scroll = scroll; r.pal = pal;
    r.ly_window = ly_window;
    render_line(r, y, line, keys, ls);
    return r.ly_window;
}

__device__ GB_NOINLINE void fill_framebuffer(uint32_t *fb, uint32_t fill) {
    for (uint32_t k = 0; k < FB_WORDS; k++) fb[k << 5] = fill;
}

// ---- deferred PPU ----------------------------------------------------------------------------------------------
// Renderer.scanline reads VRAM, OAM and the scroll / LCDC / palette registers as they are at the HBlank of the line.  The
// registers are cheap to capture; VRAM and OAM almost never change while a frame is being drawn (games update them in VBlank).
// So the emulation kernel only RECORDS the lines of the frame it has to render (lcd_record_line) and a second kernel draws
// them with one thread per (env, line) -- 144 times the parallelism of drawing inside the interpreter thread, whose dependent
// VRAM loads are pure latency.  Exactness: from the first recorded line of a frame on (defer_active) every write to VRAM / OAM
// and OAM DMA leaves the fast loop, the slow tick applies the LCD events that are due (recording their lines) and
// render_flush draws all pending lines from the still unmodified memory BEFORE the write happens.
#if defined(GB_HOSTSIM)
static unsigned long long g_hs_flushes = 0, g_hs_flushed_lines = 0;  // host harness only: how often the flush path ran
#endif
__device__ GB_NOINLINE void render_flush(Machine &m) {
#if defined(GB_HOSTSIM)
    g_hs_flushes++; g_hs_flushed_lines += m.defer_next - m.defer_from;
#endif
    for (uint32_t y = m.defer_from; y < m.defer_next; y++) {
        const uint32_t w0 = m.dl[(y * 3 + 0) << 5], w1 = m.dl[(y * 3 + 1) << 5], w2 = m.dl[(y * 3 + 2) << 5];
        render_line_out(m.memb, m.fb, w1 & 0xFF, w0, w1 >> 8, (int)w2, y, m.rline, m.rkeys, m.rls);
    }
    m.defer_from = m.defer_next = 0;
}

// HBlank of visible line y on a frame that is rendered, deferred form: capture the renderer's inputs and do its
// ly_window bookkeeping (render_line: the window line counter advances on every line that shows the window).
__device__ __forceinline__ void lcd_record_line(Machine &m, uint32_t y) {
    if (m.defer_from != m.defer_next && m.defer_next != y) render_flush(m);  // lines out of order (LCD switched off and on, LY written)
    if (m.defer_from == m.defer_next) { m.defer_from = y; }
    m.dl[(y * 3 + 0) << 5] = m.scroll;
    m.dl[(y * 3 + 1) << 5] = m.lcdc | (m.pal << 8);
    m.dl[(y * 3 + 2) << 5] = (uint32_t)m.ly_window;
    m.defer_next = y + 1;
    m.defer_active = 1;
    if ((m.lcdc & 0x20) && M_WY(m) <= y && (int)M_WX(m) - 7 < 160) m.ly_window += 1;
    if (y == 143) m.ly_window = -1;
}

__device__ __forceinline__ void lcd_blank_screen(Machine &m) {
    uint32_t shade = pal_shade(M_BGP(m), 0);
    if (m.blank_shade == shade) return;  // already uniformly this shade: the refill would be a no-op
    fill_framebuffer(m.fb, shade * 0x55555555u);
    m.blank_shade = shade;
}

// LCD.tick after `clock` has been advanced and found >= target (LCD on) or >= FRAME_CYCLES (LCD off).
__device__ inline void lcd_event(Machine &m) {
    if (m.lcdc & 0x80) {
        uint32_t irq = stat_set_mode(m, m.next_mode);
        switch (m.stat_mode) {
        case 2:
            if (m.ly == 153) {
                m.ly = 0;
                if (m.target % FRAME_CYCLES == 0) {
                    // frame-aligned LCD (the normal case): PyBoy's `clock %= 70224; target %= 70224` subtracts exactly
                    // `target` from both, whenever this event is applied (lcd_catch_up may apply it late)
                    m.cyc_adj += m.target;
                    m.clock -= m.target;
                    m.target = 0;
                } else {  // unaligned (after an LCD-off period): applied at its own tick only, see lcd_deadline
                    m.cyc_adj += m.clock - m.clock % FRAME_CYCLES;
                    m.clock %= FRAME_CYCLES;
                    m.target %= FRAME_CYCLES;
                }
            } else {
                m.ly = (m.ly + 1) & 0xFF;
            }
            m.target += 80;
            m.next_mode = 3;
            irq |= stat_update_lyc(m);
            break;
        case 3:
            m.target += 170;
            m.next_mode = 0;
            break;
        case 0:
            m.target += 206;
            if (m.ly < 144) {
                if (m.lp_dirty) {  // Renderer._scanlineparameters[y]
                    uint2 v = make_uint2(m.scroll, m.lcdc);
                    m.lp[m.ly << 5] = v;
                    m.lp_dirty--;
                }
                if (!m.disable_renderer) {
                    if (m.dl) lcd_record_line(m, m.ly);
                    else m.ly_window = render_line_out(m.memb, m.fb, m.lcdc, m.scroll, m.pal, m.ly_window, m.ly, m.rline, m.rkeys, m.rls);
                    m.blank_shade = 0xFF;
                }
            }
            m.next_mode = (m.ly < 143) ? 2 : 1;
            break;
        default:
            m.target += 456;
            m.next_mode = 1;
            m.ly = (m.ly + 1) & 0xFF;
            irq |= stat_update_lyc(m);
            if (m.ly == 144) {
                irq |= IRQ_VBLANK;
                m.frame_done = 1;
                m.defer_active = 0;  // the frame's pending lines are drawn after the kernel (or at the start of its next frame)
            }
            if (m.ly == 153) m.next_mode = 2;
            break;
        }
        m.iflag |= irq;
    } else {
        m.frame_done = 1;
        m.cyc_adj += m.clock - m.clock % FRAME_CYCLES;
        m.clock %= FRAME_CYCLES;
        m.defer_from = m.defer_next = m.defer_active = 0;  // whatever was pending is painted over
        lcd_blank_screen(m);
    }
}

// ---- lazy LCD ------------------------------------------------------------------------------------------------
// PyBoy's LCD.tick changes mode 442 times a frame, but while no STAT interrupt source is armed only two kinds of
// mode change have effects outside the LCD's own registers: entering VBlank (IF bit 0, end of Motherboard.tick's frame)
// and, on a frame whose renderer is enabled, the HBlank of a visible line (Renderer.scanline reads VRAM / OAM / the
// scroll registers as they are at that moment).  Every other mode change ("soft") only rewrites LY, STAT's mode / LYC
// bits, clock_target and the saved scanline parameters -- state nothing can see without a bus access.  So the interpreter
// runs to the next HARD event (lcd_deadline) and the soft ones in between are applied, in order and with exactly the
// effects LCD.tick would have had, by lcd_catch_up: at the deadline, and before any bus access that could observe or
// change LCD state (every out-of-line read or write).  With a STAT source armed or TIMA running (a halted CPU then
// ticks the timer once per LCD event) every event is hard and this degenerates to PyBoy's one-event-per-tick loop.

// Cycles from lcd.clock to the next hard event; records in m.lazy whether soft events may be applied late.
__device__ GB_NOINLINE int lcd_deadline(Machine &m) {
    m.lazy = 0;
    if (!(m.lcdc & 0x80)) return (int)(FRAME_CYCLES - m.clock);
    const int t = (int)(m.target - m.clock);
    // t <= 0: an event is already due (only inconsistent loaded states get here): strict one event per tick
    if ((m.stat & 0x78) | (m.tmr & 0x04000000u) | (uint32_t)(t <= 0)) return t;
    const uint32_t nm = m.next_mode, ly = m.ly;
    // no line of this frame needs the renderer at its HBlank: rendering is off, or the lines are only recorded (deferred PPU; the
    // first one of a frame is still a hard event: it arms defer_active, which sends VRAM / OAM writes through the slow tick)
    const bool no_draw = m.disable_renderer || (m.dl && m.defer_active);
    int d;
    if (nm == 1) {
        if (ly == 143) return t;           // the next event enters VBlank
        if (ly - 144u > 8u) return t;      // inconsistent state: not lazy
        // in VBlank: LY 153 -> 0 is `153 - ly` events away.  Its clock wrap can only be applied late when the frame is
        // aligned (lcd_event); otherwise stop there.
        const int wrap = t + 456 * (int)(153 - ly);
        if ((m.target + 456u * (153 - ly)) % FRAME_CYCLES != 0) { m.lazy = 1; return wrap; }
        d = no_draw ? wrap + 456 * 144 : wrap + 250;
    } else if (nm == 2) {
        if (ly == 153) {
            if (m.target % FRAME_CYCLES != 0) return t;
            d = no_draw ? t + 456 * 144 : t + 250;
        } else {
            if (ly > 142) return t;
            d = no_draw ? t + 456 * (int)(143 - ly) : t + 250;
        }
    } else {
        if (ly > 143) return t;
        const int to_hblank = nm == 3 ? t + 170 : t;  // mode 2 -> 3 -> 0
        d = no_draw ? to_hblank + 206 + 456 * (int)(143 - ly) : to_hblank;
    }
    m.lazy = 1;
    return d;
}

// Applies every LCD event that is due (clock >= clock_target).  Not lazy: exactly one, as LCD.tick does per CPU tick.
__device__ GB_NOINLINE void lcd_catch_up(Machine &m) {
    if (!(m.lcdc & 0x80)) {
        if (m.clock >= FRAME_CYCLES) lcd_event(m);
        return;
    }
    const uint32_t lazy = m.lazy;
    while ((int)(m.clock - m.target) >= 0) {
        const uint32_t behind = m.clock - m.target;
        const bool recording = !m.disable_renderer && m.dl && m.defer_active;
        if (lazy && (m.disable_renderer || recording) && m.stat_mode == 0 && m.next_mode == 2 && m.ly < 142 && behind >= 456) {
            // whole visible lines without drawing: mode 2 / 3 / 0 of each only move LY, STAT, clock_target, the saved scanline
            // parameters and (deferred PPU) the line records -- closed form for k lines, staying below line 143 (whose HBlank
            // arms the VBlank entry)
            uint32_t k = behind / 456;
            if (k > 142 - m.ly) k = 142 - m.ly;
            for (uint32_t y = m.ly + 1; y <= m.ly + k && (m.lp_dirty || recording); y++) {
                if (m.lp_dirty) {
                    m.lp[y << 5] = make_uint2(m.scroll, m.lcdc);
                    m.lp_dirty--;
                }
                if (recording) lcd_record_line(m, y);
            }
            m.ly += k;
            m.stat = (m.stat & 0xF8) | (m.lyc == m.ly ? 0x04 : 0);
            m.target += 456 * k;
            continue;
        }
        lcd_event(m);
        if (!lazy) break;
    }
}

// ------------------------------------------------------------------------------------------- timer

__device__ __forceinline__ uint32_t timer_divider(uint32_t tac) {
    return (tac & 3) == 0 ? 1024u : (4u << ((tac & 3) * 2));  // 1024, 16, 64, 256
}

// Timer.tick, TIMA half (PyBoy: one increment per tick at most).  The DIV half is `divc += cycles`, which the
// interpreter applies lazily together with the LCD clock (DIV = div + (divc >> 8), materialised on read / store).
__device__ __forceinline__ void timer_tick_tima(Machine &m, uint32_t cycles) {
    if (m.tmr & 0x04000000u) {  // TAC bit 2: timer enabled
        m.timac += cycles;
        uint32_t dv = timer_divider(M_TAC(m));
        if (m.timac >= dv) {
            m.timac -= dv;
            if (M_TIMA(m) == 0xFF) {
                m.tmr = (m.tmr & 0xFFFF00FFu) | (M_TMA(m) << 8);
                m.iflag |= IRQ_TIMER;
            } else {
                m.tmr += 0x100;
            }
        }
    }
}

__device__ __forceinline__ int timer_cycles_to_interrupt(const Machine &m) {
    if (!(m.tmr & 0x04000000u)) return 1 << 16;
    return (int)((0x100 - M_TIMA(m)) * timer_divider(M_TAC(m))) - (int)m.timac;
}

// --------------------------------------------------------------------------------------------- bus
// The interpreter (gb_cpu.cuh) defers all stores of an instruction to one write site; its read and write
// sites inline only the hot regions (WRAM, ROM, HRAM, VRAM, OAM); IO registers, MBC
// registers, cart RAM and OAM DMA live in out-of-line functions that take their inputs BY VALUE (reads) or
// work on a scratch copy of the machine (writes), so `Machine` itself never has its address taken and
// stays in registers, and the hot loop stays small (the kernel is instruction-cache sensitive).

#define IO_NOT_A_REGISTER 0x100u
// value of an IO register modelled outside the IO array, or IO_NOT_A_REGISTER
__device__ GB_NOINLINE uint32_t io_reg_read(uint32_t a, uint32_t lcd0 /* LCDC STAT LY LYC */, uint32_t scroll /* SCX SCY WX WY */,
                                             uint32_t pal_ie /* BGP OBP0 OBP1 IE */, uint32_t tim /* DIV TIMA TMA TAC */, uint32_t iflag) {
    switch (a) {
    case 0xFF04: return tim & 0xFF;
    case 0xFF05: return (tim >> 8) & 0xFF;
    case 0xFF06: return (tim >> 16) & 0xFF;
    case 0xFF07: return tim >> 24;
    case 0xFF0F: return iflag;
    case 0xFF40: return lcd0 & 0xFF;
    case 0xFF41: return (lcd0 >> 8) & 0xFF;
    case 0xFF42: return (scroll >> 8) & 0xFF;
    case 0xFF43: return scroll & 0xFF;
    case 0xFF44: return (lcd0 >> 16) & 0xFF;
    case 0xFF45: return lcd0 >> 24;
    case 0xFF46: return 0;
    case 0xFF47: return pal_ie & 0xFF;
    case 0xFF48: return (pal_ie >> 8) & 0xFF;
    case 0xFF49: return (pal_ie >> 16) & 0xFF;
    case 0xFF4A: return scroll >> 24;
    case 0xFF4B: return (scroll >> 16) & 0xFF;
    case 0xFFFF: return pal_ie >> 24;
    default: return (a >= 0xFF10 && a < 0xFF40) ? 0u : IO_NOT_A_REGISTER;  // sound disabled (pokegym default): reads 0
    }
}

__device__ __forceinline__ uint32_t bus_read_full(Machine &m, uint32_t a) {  // Motherboard.getitem
    if (a - 0xC000u < 0x3E00u) return mem_rd(m, MEM_WRAM + (a & 0x1FFF));  // WRAM and its echo
    if (a < 0x8000) return __ldg(m.rom + (a < 0x4000 ? a : a + m.rom_off));
    if (a >= 0xFF80 && a != 0xFFFF) return mem_rd(m, MEM_HI + (a - 0xFE00));  // HRAM
    if (a < 0xA000) return mem_rd(m, MEM_VRAM + (a - 0x8000));
    if (a < 0xC000) {
        if (!m.ram_en) return 0xFF;
        uint32_t i = (m.rambank & 3) * 0x2000u + (a - 0xA000);
        return m.cramb[((i >> 2) << 7) | (i & 3)];
    }
    if (a >= 0xFF00) {
        uint32_t r = io_reg_read(a, m.lcdc | (m.stat << 8) | (m.ly << 16) | (m.lyc << 24), m.scroll, m.pal | (m.ie << 24),
                                 ((m.div + (m.divc >> 8)) & 0xFF) | m.tmr, m.iflag);
        if (r != IO_NOT_A_REGISTER) return r;
    }
    return mem_rd(m, MEM_HI + (a - 0xFE00));  // OAM, 0xFEA0-0xFEFF, plain IO array bytes
}
__device__ GB_NOINLINE uint32_t bus_read_slow(Machine &m, uint32_t a) { return bus_read_full(m, a); }
__device__ __forceinline__ uint32_t bus_read(Machine &m, uint32_t a) {  // wrapper kernels / debug access
    if (a < 0x8000) return __ldg(m.rom + (a < 0x4000 ? a : a + m.rom_off));
    if (a >= 0xC000 && a < 0xE000) return mem_rd(m, MEM_WRAM + (a - 0xC000));
    return bus_read_slow(m, a);
}

// Everything a store can do besides hitting plain RAM: MBC3 registers, cart RAM, IO registers, OAM DMA.
__device__ GB_NOINLINE void bus_write_rare(Machine *mp, uint32_t a, uint32_t v) {
    Machine &m = *mp;
    if (a < 0x8000) {  // MBC3 registers
        if (a < 0x2000) {
            if ((v & 0x0F) == 0x0A) m.ram_en = 1;
            else if (v == 0) m.ram_en = 0;  // PyBoy: any other value leaves the latch untouched
        } else if (a < 0x4000) {
            v &= 0x7F;
            machine_set_rombank(m, v ? v : 1);
        } else if (a < 0x6000) {
            m.rambank = v;
        }
        return;
    }
    if (a < 0xA000) { mem_wr(m, MEM_VRAM + (a - 0x8000), v); return; }
    if (a < 0xC000) {  // 0xA000-0xBFFF cart RAM
        if (m.ram_en && m.rambank <= 3) {
            uint32_t i = m.rambank * 0x2000u + (a - 0xA000);
            m.cramb[((i >> 2) << 7) | (i & 3)] = (uint8_t)v;
        }
        return;
    }
    if (a < 0xFE00) { mem_wr(m, MEM_WRAM + (a & 0x1FFF), v); return; }  // WRAM / echo (only reached through bus_write)
    if (a < 0xFF00 || (a >= 0xFF80 && a != 0xFFFF)) { mem_wr(m, MEM_HI + (a - 0xFE00), v); return; }
    switch (a) {
    case 0xFF00: mem_wr(m, MEM_HI + 0x100, joypad_pull(m, v)); break;
    case 0xFF04: m.div = 0; m.divc = 0; m.timac = 0; break;
    case 0xFF05: m.tmr = (m.tmr & 0xFFFF00FFu) | (v << 8); break;
    case 0xFF06: m.tmr = (m.tmr & 0xFF00FFFFu) | (v << 16); break;
    case 0xFF07: m.tmr = (m.tmr & 0x00FFFFFFu) | ((v & 7) << 24); break;
    case 0xFF0F: m.iflag = v; break;
    case 0xFF40: lcd_set_lcdc(m, v); break;
    case 0xFF41: m.stat = (m.stat & 0x87) | (v & 0x78); break;
    case 0xFF42: if (v != M_SCY(m)) m.lp_dirty = 144; m.scroll = (m.scroll & 0xFFFF00FFu) | (v << 8); break;
    case 0xFF43: if (v != M_SCX(m)) m.lp_dirty = 144; m.scroll = (m.scroll & 0xFFFFFF00u) | v; break;
    case 0xFF44: m.ly = v; m.lp_dirty = 144; break;  // PyBoy lets LY be written
    case 0xFF45: m.lyc = v; break;
    case 0xFF46: {  // Motherboard.transfer_DMA: instantaneous copy of 0xA0 bytes to OAM
        uint32_t src = v << 8;
        bool plain = (v >= 0x80 && v < 0xA0) || (v >= 0xC0 && v < 0xFE);
        if (plain) {  // word copy inside the plain-RAM array (src is 256-byte aligned)
            uint32_t base = v < 0xA0 ? (MEM_VRAM + (src - 0x8000)) : (MEM_WRAM + (src & 0x1FFF));
            for (uint32_t k = 0; k < 40; k++) mem_wr_word(m, (MEM_HI >> 2) + k, mem_rd_word(m, (base >> 2) + k));
        } else {
            for (uint32_t k = 0; k < 160; k++) mem_wr(m, MEM_HI + k, bus_read_full(m, (src + k) & 0xFFFF));
        }
        break;
    }
    case 0xFF47: m.pal = (m.pal & 0xFFFF00u) | v; break;
    case 0xFF48: m.pal = (m.pal & 0xFF00FFu) | (v << 8); break;
    case 0xFF49: m.pal = (m.pal & 0x00FFFFu) | (v << 16); break;
    case 0xFF4A: if (v != M_WY(m)) m.lp_dirty = 144; m.scroll = (m.scroll & 0x00FFFFFFu) | (v << 24); break;
    case 0xFF4B: if (v != M_WX(m)) m.lp_dirty = 144; m.scroll = (m.scroll & 0xFF00FFFFu) | (v << 16); break;
    case 0xFFFF: m.ie = v; break;
    default:
        if (a >= 0xFF10 && a < 0xFF40) break;  // sound disabled: writes dropped
        mem_wr(m, MEM_HI + (a - 0xFE00), v);
        break;
    }
}

__device__ __forceinline__ void bus_write_full(Machine &m, uint32_t a, uint32_t v) {  // Motherboard.setitem
    v &= 0xFF;
    if (a - 0xC000u < 0x3E00u) { mem_wr(m, MEM_WRAM + (a & 0x1FFF), v); return; }
    if (a >= 0xFF80 && a != 0xFFFF) { mem_wr(m, MEM_HI + (a - 0xFE00), v); return; }
    // deferred PPU: recorded lines are drawn from VRAM / OAM as they are NOW, before this write changes them
    if (m.defer_from != m.defer_next && (a - 0x8000u < 0x2000u || a - 0xFE00u < 0x100u || a == 0xFF46u)) render_flush(m);
    if (a >= 0xFE00 && a < 0xFF00) { mem_wr(m, MEM_HI + (a - 0xFE00), v); return; }
    if (a - 0x8000u < 0x2000u) { mem_wr(m, MEM_VRAM + (a - 0x8000), v); return; }
    bus_write_rare(&m, a, v);
}
__device__ __forceinline__ void bus_write(Machine &m, uint32_t a, uint32_t v) {  // wrapper kernels / debug access
    v &= 0xFF;
    if (a >= 0xC000 && a < 0xE000) mem_wr(m, MEM_WRAM + (a - 0xC000), v);
    else bus_write_full(m, a, v);
}

// ------------------------------------------------------------------------------------------- SM83

__device__ __forceinline__ uint32_t reg8(const Machine &m, uint32_t idx) {  // B C D E H L - A
    uint32_t w = (idx & 4) ? m.hlaf : m.bcde;
    return (w >> (((idx ^ 1) & 3) * 8)) & 0xFF;
}
__device__ __forceinline__ void set_reg8(Machine &m, uint32_t idx, uint32_t v) {
    uint32_t sh = ((idx ^ 1) & 3) * 8, mask = 0xFFu << sh;
    if (idx & 4) m.hlaf = (m.hlaf & ~mask) | ((v & 0xFF) << sh);
    else m.bcde = (m.bcde & ~mask) | ((v & 0xFF) << sh);
}
__device__ __forceinline__ uint32_t reg_a(const Machine &m) { return (m.hlaf >> 16) & 0xFF; }
__device__ __forceinline__ uint32_t reg_f(const Machine &m) { return m.hlaf >> 24; }
__device__ __forceinline__ uint32_t reg_hl(const Machine &m) { return m.hlaf & 0xFFFF; }
__device__ __forceinline__ void set_a(Machine &m, uint32_t v) { m.hlaf = (m.hlaf & 0xFF00FFFFu) | ((v & 0xFF) << 16); }
__device__ __forceinline__ void set_f(Machine &m, uint32_t v) { m.hlaf = (m.hlaf & 0x00FFFFFFu) | (v << 24); }
__device__ __forceinline__ void set_af(Machine &m, uint32_t a, uint32_t f) { m.hlaf = (m.hlaf & 0xFFFFu) | ((a & 0xFF) << 16) | (f << 24); }
__device__ __forceinline__ void set_hl(Machine &m, uint32_t v) { m.hlaf = (m.hlaf & 0xFFFF0000u) | (v & 0xFFFF); }
__device__ __forceinline__ uint32_t reg_pair(const Machine &m, uint32_t p) {  // BC DE HL SP
    return p == 0 ? (m.bcde & 0xFFFF) : p == 1 ? (m.bcde >> 16) : p == 2 ? (m.hlaf & 0xFFFF) : m.sp;
}
__device__ __forceinline__ void set_reg_pair(Machine &m, uint32_t p, uint32_t v) {
    v &= 0xFFFF;
    if (p == 0) m.bcde = (m.bcde & 0xFFFF0000u) | v;
    else if (p == 1) m.bcde = (m.bcde & 0xFFFFu) | (v << 16);
    else if (p == 2) m.hlaf = (m.hlaf & 0xFFFF0000u) | v;
    else m.sp = v;
}
__device__ __forceinline__ bool condition(const Machine &m, uint32_t cc) {  // NZ Z NC C
    uint32_t f = reg_f(m);
    uint32_t bit = (cc & 2) ? (f & FLAG_C) : (f & FLAG_Z);
    return (bit != 0) == ((cc & 1) != 0);
}

// 8-bit ALU group (ADD ADC SUB SBC AND XOR OR CP) on A with operand v.  Branch-free: in this kernel a divergent
// region costs about as much as twenty ALU instructions, and lanes running different ALU ops stay converged.
// Subtraction is addition of the complement with inverted carry-in; its H and C flags are the inverted carries.
__device__ __forceinline__ void alu8(Machine &m, uint32_t op, uint32_t v) {
    const uint32_t a = reg_a(m), carry = (reg_f(m) >> 4) & 1;
    const bool logic = (op - 4u) < 3u;             // AND XOR OR
    const bool sub = (op == 2) | (op == 3) | (op == 7);  // SUB SBC CP
    const uint32_t cin = (op & 1) & (op < 4) ? carry : 0;   // ADC / SBC only
    const uint32_t x = sub ? (v ^ 0xFF) : v, c0 = sub ? (cin ^ 1) : cin;
    const uint32_t sum = a + x + c0;
    const uint32_t hc = (((a & 0xF) + (x & 0xF) + c0) >> 4) & 1, cc = (sum >> 8) & 1;  // carries out of bit 3 / bit 7
    const uint32_t lres = op == 4 ? (a & v) : op == 5 ? (a ^ v) : (a | v);
    const uint32_t res = logic ? lres : (sum & 0xFF);
    uint32_t nf = logic ? (op == 4 ? FLAG_H : 0) : (((hc ^ (uint32_t)sub) ? FLAG_H : 0) | ((cc ^ (uint32_t)sub) ? FLAG_C : 0) | (sub ? FLAG_N : 0));
    if (res == 0) nf |= FLAG_Z;
    set_af(m, op == 7 ? a : res, nf);
}
