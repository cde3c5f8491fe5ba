// gb_cpu.cuh -- SM83 interpreter of k_run_frames (CPU.tick of PyBoy 1.6: interrupt check, HALT, one instruction,
// then the peripherals advance by its T-cycles; interrupt dispatch costs 0 cycles).
//
// Design (B200-first; nothing here resembles a CPU interpreter's fetch/decode/execute switch):
//   * The env's whole `Machine` lives in SHARED memory; only what every instruction touches is cached in registers:
//     the two packed register words, SP, PC, the ROM bank offset, a cycle countdown and a 2-bit mode word.
//   * Two instantiations of ONE instruction body (cpu_exec<FAST>).  The hot loop of cpu_run_to_event is the FAST one
//     and contains no call at all: code in ROM or HRAM, reads of WRAM / HRAM / ROM, writes to WRAM / HRAM / OAM / VRAM and
//     the MBC3 bank-select register.  Whatever else an instruction needs -- an IO register, cart RAM, a rare opcode,
//     interrupt dispatch, HALT, a running TIMA -- makes the fast body decline BEFORE it has changed anything, and the
//     tick is redone from scratch by cpu_tick_slow, an out-of-line function that works on the parked machine with full
//     bus semantics.  One call site means no hot value is live across a call and no convergence-barrier state to save.
//   * One 128-bit read-only load fetches the pre-decoded control word of the instruction (gb_predecode.h).  Operand
//     fetch (register byte by PRMT, immediate, or ONE shared copy of the bus read), register write-back (two PRMTs
//     with ready-made selectors) and the deferred bus write are the same straight-line code for all instructions, so
//     lanes of a warp that execute different instructions stay converged everywhere except inside the short handler
//     bodies, which the switch groups by handler id (lanes with the same id run together, whatever their PC).
//   * Time is ONE register: `rem` = cycles until this env's next LCD mode change.  lcd.clock and the DIV counter are
//     brought up to date (time_sync) only when something observes them.
#pragma once
#include "gb_device.cuh"
#include "gb_predecode.h"

// The fast loop exists in two builds, selected by the template parameter SIMT:
//   SIMT = true  (k_run_frames, several envs per warp): whatever makes the instruction body decline only sets a flag and the
//                one exit sits in front of the write-back.  Every divergent region is then single-entry / single-exit, nvcc
//                gives each a re-convergence point, and the write-back, the stores and the loop tail run once per warp
//                instead of once per handler group (measured before: 2.5 executions per iteration with 2.9 of 8 lanes).
//   SIMT = false (k_run_frames_1, one env per single-thread block): declines return at once -- fewer instructions, and there
//                is nothing to re-converge.
// Measured on B200 (tools/gpu_variants.sh, env-steps/s): 4,096 envs, 1 lane: 127.0 k early-return / 120.8 k flag;
// 32,768 envs, 16 lanes: 502 k early-return / 552 k flag; an explicit __syncwarp in front of the write-back added nothing
// to the flag build (554 k) and cost 9 % at 1 lane.  One body for ROM + HRAM code and flag-bit dispatch of INC/DEC and the
// arithmetic group help both (+4 % / +7 %).
#if !defined(GB_TRACE_SLOT)
#define GB_TRACE_SLOT(kind, phys, dx, dw)  // host-side convergence study only (tests/hostsim, -DGB_SLOT_TRACE)
#endif

__constant__ uint4 c_base_desc[512];  // per-opcode base descriptors (pd_build_base), uploaded once per process

#define MODE_ATTN 0x8000u   // pending interrupt / HALT / PyBoy's interrupt_queued latch: the tick starts in cpu_attention
#define MODE_POST 0x10000u  // HALT: the tick ends in cpu_post_slow
#define MODE_DEFER 0x20000u  // deferred PPU: a line of this frame is recorded -- VRAM / OAM stores go through the slow tick (render_flush)

struct RunCtx {  // uniform per launch
    const uint4 *rom_dec;
    uint32_t bank_mask;  // rom_banks - 1 when that is a power of two, else 0
};

__device__ __forceinline__ uint32_t hot_mode(const Machine &m) {
    const uint32_t attn = m.halted | m.iq | (m.iflag & m.ie & 0x1F), post = m.halted;
    return (attn ? MODE_ATTN : 0u) | (post ? MODE_POST : 0u) | (m.defer_active ? MODE_DEFER : 0u);
}
#define TIMA_ON 0x04000000u  // TAC bit 2 inside Machine.tmr
// Cycles until the interpreter has to stop: for the LCD (the next hard event, see lcd_deadline) or, while TIMA runs, for the
// tick in which Timer.tick's counter reaches the divider (PyBoy: one TIMA increment per CPU tick at most, so a counter that
// is already past the divider fires again on the very next tick).
// `fresh`: no executed tick is waiting for its share of the countdown: a counter already past the divider fires with the NEXT
// tick (one instruction is let through).  After a slow tick (!fresh) the caller subtracts that tick's cycles, and a result <= 0
// means that very tick fires -- also a 0-cycle interrupt dispatch on a counter that is past the divider.
__device__ __forceinline__ int hot_rem(Machine &m, bool fresh) {
    int rem = lcd_deadline(m);
    if (m.tmr & TIMA_ON) {
        int rt = (int)timer_divider(M_TAC(m)) - (int)m.timac;
        if (fresh) rt = rt < 1 ? 1 : rt;
        rem = rt < rem ? rt : rem;
    }
    return rem;
}
// bring lcd.clock, the DIV counter and (while TIMA runs) Timer.tick's TIMA counter up to the interpreter's countdown
__device__ __forceinline__ void time_sync(Machine &m, int rem) {
    const uint32_t e = (uint32_t)(m.t_sync - rem);
    m.clock += e;
    m.divc += e;
    if (m.tmr & TIMA_ON) m.timac += e;
    m.t_sync = rem;
}

// one thread per ROM offset
__global__ void k_predecode_rom(const uint8_t *rom, uint32_t rom_len, uint4 *out) {
    uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= rom_len) return;
    uint32_t in_bank = o & 0x3FFF;
    if (in_bank >= 0x3FFD) {  // operands would come from another bank: decode at run time
        out[o] = make_uint4(H_SLOW, 0, 0x32103210u, PD_NO_CLASS_W);
        return;
    }
    uint32_t ins = rom[o] | (rom[o + 1] << 8) | (rom[o + 2] << 16);
    out[o] = pd_finish(c_base_desc[(ins & 0xFF) == 0xCB ? (256u | ((ins >> 8) & 0xFF)) : (ins & 0xFF)], ins, o < 0x4000 ? o : 0x4000 + in_bank);
}

// Decode at run time: RAM-resident code and the last three bytes of a ROM bank.  HRAM (where every game keeps its
// OAM-DMA stub, ~80 instructions per frame) is read as two aligned words; everything else goes byte-wise through the bus.
__device__ GB_NOINLINE uint4 cpu_decode_slow(Machine &m, uint32_t pc) {
    uint32_t ins = 0;
    if (pc - 0xFF80u < 0x7Du) {
        const uint32_t i = MEM_HI + (pc - 0xFE00), w0 = mem_rd_word(m, i >> 2), w1 = mem_rd_word(m, (i >> 2) + 1), sh = (i & 3) * 8;
        ins = sh ? ((w0 >> sh) | (w1 << (32 - sh))) : w0;
    } else {
        for (uint32_t i = 0; i < 3; i++) ins |= bus_read_full(m, (pc + i) & 0xFFFF) << (8 * i);
    }
    return pd_finish(c_base_desc[(ins & 0xFF) == 0xCB ? (256u | ((ins >> 8) & 0xFF)) : (ins & 0xFF)], ins, pc);
}

// Start of a tick that needs attention (CPU.tick / CPU.check_interrupts / CPU.handle_interrupt of PyBoy 1.6).
// Works on the spilled machine.  Returns 1 when an instruction is to be executed, else (T-cycles << 8).
__device__ GB_NOINLINE uint32_t cpu_attention(Machine &m) {
    if (!m.iq) {
        const uint32_t pending = m.iflag & m.ie & 0x1F;
        if (pending) {  // highest-priority pending source
            const uint32_t bit = pending & (0u - pending);
            if (m.halted) m.pc = (m.pc + 1) & 0xFFFF;
            if (m.ime) {
                m.iflag ^= bit;
                bus_write_full(m, (m.sp - 1) & 0xFFFF, m.pc >> 8);
                bus_write_full(m, (m.sp - 2) & 0xFFFF, m.pc & 0xFF);
                m.sp = (m.sp - 2) & 0xFFFF;
                m.pc = 0x40 + 8 * (31 - __clz(bit));
                m.ime = 0;
            }
            m.iq = 1;
            m.halted = 0;
            return 0;  // dispatch costs no cycles and executes nothing
        }
    } else if (m.halted) {  // debugger-only path in PyBoy: halted with a queued interrupt
        m.halted = 0;
        m.pc = (m.pc + 1) & 0xFFFF;
    }
    if (m.halted) return 4u << 8;
    m.iq = 0;
    return 1;
}

// End of a tick while halted or with TIMA running: HALT fast-forward (Motherboard.tick) and Timer.tick's TIMA half.
__device__ GB_NOINLINE uint32_t cpu_post_slow(Machine &m, uint32_t cycles) {
    if (m.halted) {  // fast-forward to the next (hard) LCD event / timer overflow
        // PyBoy: min(lcd.clock_target - lcd.clock, timer.cycles_to_interrupt()), i.e. the halted CPU ticks once per LCD
        // mode change.  While nothing is pending it just halts again, so the ticks up to the next *hard* event collapse
        // into one; with an interrupt already pending (IF & IE) the very next tick ends the HALT, at the next mode change.
        const bool sleeps_on = (m.lcdc & 0x80) && !(m.iflag & m.ie & 0x1F);
        const int a = sleeps_on ? lcd_deadline(m) : (int)(m.target - m.clock), b = timer_cycles_to_interrupt(m), c = a < b ? a : b;
        cycles = c < 0 ? 0u : (uint32_t)c;
        if ((m.tmr & 0x04000000u) && b <= 0 && !(m.iflag & m.ie & 0x1F)) {
            // The TIMA counter is so far past the divider that the timer interrupt is "due" (PyBoy: cycles_to_interrupt <= 0):
            // the halted CPU now spins through 0-cycle ticks, each incrementing TIMA once, until TIMA overflows -- nothing else
            // changes meanwhile (no cycles pass, nothing is pending).  All but the last of those 0x100 - TIMA ticks are applied
            // here in closed form; the last one, the overflow, is the timer_tick_tima below.
            const uint32_t n = 0xFFu - M_TIMA(m);
            m.timac -= n * timer_divider(M_TAC(m));
            m.tmr |= 0xFF00u;
        }
    }
    timer_tick_tima(m, cycles);
    return cycles;
}


struct CpuRegs {
    uint32_t bcde, hlaf, sp, pc;
};

// What the fast body may touch without leaving the loop.
// Byte offset inside the env's interleaved plain-RAM array of a store the fast body may do itself, 0xFFFFFFFE for a store
// that is dropped (sound registers: PyBoy with sound disabled, pokegym's configuration, ignores them), 0xFFFFFFFD for the
// MBC3 ROM-bank register, or 0xFFFFFFFF when the store needs the full bus (IO, other MBC registers, cart RAM).
#define FAST_WR_NONE 0xFFFFFFFFu
#define FAST_WR_DROP 0xFFFFFFFEu
#define FAST_WR_BANK 0xFFFFFFFDu
#define FAST_WR_P1 0xFFFFFFFCu  // the joypad select register: the stored byte is Interaction.pull of the written one
__device__ __forceinline__ uint32_t mem_offset(uint32_t i) { return ((i >> 2) << 7) | (i & 3); }
__device__ __forceinline__ uint32_t fast_store_target(uint32_t a) {  // single-lane build: first match wins
    if (a - 0xC000u < 0x3E00u) return mem_offset(MEM_WRAM + (a & 0x1FFF));                               // WRAM and its echo
    if (a - 0xFF80u < 0x7Fu || a - 0xFE00u < 0x100u) return mem_offset(MEM_HI + (a - 0xFE00));             // HRAM, OAM
    if (a - 0x8000u < 0x2000u) return mem_offset(MEM_VRAM + (a - 0x8000));                                // VRAM
    if (a - 0x2000u < 0x2000u) return FAST_WR_BANK;
    if (a - 0xFF10u < 0x30u) return FAST_WR_DROP;
    if (a == 0xFF00u) return FAST_WR_P1;
    return FAST_WR_NONE;
}
// Plain RAM behind address `a`: work RAM and its echo, VRAM, OAM / 0xFEA0-0xFEFF, HRAM (0xFF80-0xFFFE).  Returns whether it
// is, and the byte offset inside the env's interleaved array (meaningless otherwise).  Selects only.
__device__ __forceinline__ bool fast_plain_offset(uint32_t a, uint32_t &off) {
    const bool wram = a - 0xC000u < 0x3E00u, vram = a - 0x8000u < 0x2000u;
    const bool hi = (a - 0xFE00u < 0x100u) | (a - 0xFF80u < 0x7Fu);
    const uint32_t i = wram ? MEM_WRAM + (a & 0x1FFF) : a + (vram ? MEM_VRAM - 0x8000u : MEM_HI - 0xFE00u);
    off = mem_offset(i);
    return wram | vram | hi;
}
// byte at base + off when `ok`, else `otherwise`: a predicated load (no branch: the lanes of a warp stay together whatever
// kind of memory each of them reads)
__device__ __forceinline__ uint32_t fast_load_u8(const uint8_t *base, uint32_t off, bool ok, uint32_t otherwise) {
#if defined(GB_HOSTSIM)
    return ok ? base[off] : otherwise;
#else
    uint32_t r = otherwise;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p ld.global.u8 %0, [%1];\n\t}" : "+r"(r) : "l"(base + off), "r"((uint32_t)ok) : "memory");
    return r;
#endif
}
// both bytes of a push below `sp` inside work RAM (or its echo)
__device__ __forceinline__ bool fast_stack_push(uint32_t sp) { return sp - 0xC002u < 0x3DFFu; }

// One instruction, given its control word.  FAST: returns false -- having changed nothing -- when the instruction needs
// anything outside the fast set; `mode` is only read.  !FAST: always completes (full bus, every opcode).
// Outputs: r (registers incl. pc), rom_off (bank switches), cyc, mode (HALT).
// FAST && SIMT: `declined` may come in already set (no descriptor could be fetched); the body has no exit in front of the
// write-back.
template <bool FAST, bool SIMT, int CH = -1, uint32_t CF = 0>
__device__ __forceinline__ bool cpu_exec(Machine &m, const uint4 d, CpuRegs &r, uint32_t &rom_off, uint32_t &mode, uint32_t &cyc, uint8_t *memb,
                                         const uint8_t *rom, uint32_t bank_mask, bool declined = false) {
    uint32_t bcde = r.bcde, hlaf = r.hlaf, sp = r.sp;
#define FAST_DECLINE()         \
    do {                       \
        if (!SIMT) return false; \
        declined = true;       \
    } while (0)
    auto rd8 = [&](uint32_t a) -> uint32_t {  // Motherboard.getitem; FAST: WRAM (+ echo), ROM and HRAM, else decline
        if (FAST) {
            if (a - 0xC000u < 0x3E00u) return memb[mem_offset(MEM_WRAM + (a & 0x1FFF))];
            if (a < 0x8000u) return __ldg(rom + (a + (a >> 14) * rom_off));
            if (a - 0xFF80u < 0x7Fu || a - 0xFF00u < 4u) return memb[mem_offset(MEM_HI + (a - 0xFE00))];  // HRAM; P1, SB, SC
            declined = true;
            return 0;
        }
        return bus_read_full(m, a);
    };
    // ---- operand fetch (uniform)
    // CH >= 0: an instance for ONE class of instruction (gb_classes.inc) -- handler id and operand flags are compile-time
    // constants, every test on them below folds away; CH < 0: the generic body, both come from the control word
    const uint32_t w = d.w, wf = CH >= 0 ? CF : d.w, h = CH >= 0 ? (uint32_t)CH : (d.x & 0xFF);
    uint32_t v = gb_prmt(bcde, hlaf, w);  // byte 0 = source register (upper bytes: don't care)
    if (wf & PDF_IMM) v = d.y & 0xFFFFu;
    uint32_t wa = 0, wt = 0;  // store address; FAST: its classified target
    // FAST: whatever makes the body decline only sets `declined`; the one exit is in front of the write-back, so every
    // divergent region below is single-entry / single-exit and the lanes of a warp re-converge behind each of them
    // (rare opcodes and descriptors that could not be pre-decoded carry no operand flags: the fast body finds out in the
    // handler switch's default case, having changed nothing -- one test less on every other instruction)
    if (wf & (PDF_RD | PDF_WR)) {
        wa = (wf & PDF_AIMM) ? (d.y & 0xFFFFu) : (gb_prmt(bcde, hlaf, w >> 16) & 0xFFFFu);
        if (wf & PDF_ASP) wa = sp;
        if (FAST && SIMT) {
            // ONE straight-line classification of the address serves the read and the deferred store: plain RAM (work RAM
            // and its echo, VRAM, OAM / 0xFEA0-0xFEFF, HRAM -- Motherboard.getitem / setitem touch nothing else for these)
            // is an offset into this env's interleaved array, ROM a pointer into the shared image; selects, no branches
            uint32_t off;
            const bool plain = fast_plain_offset(wa, off);
            if (wf & PDF_WR) {
                wt = plain ? off : (wa - 0x2000u < 0x2000u) ? FAST_WR_BANK : (wa - 0xFF10u < 0x30u) ? FAST_WR_DROP : wa == 0xFF00u ? FAST_WR_P1 : FAST_WR_NONE;
                if (wt == FAST_WR_NONE) FAST_DECLINE();
                if ((mode & MODE_DEFER) && (wa - 0x8000u < 0x2000u || wa - 0xFE00u < 0x100u)) FAST_DECLINE();  // render_flush first
            }
            if (wf & PDF_RD) {
                // P1 (the byte Interaction.pull left there), SB, SC and 0xFF03 read back from the IO array like plain RAM
                const bool in_rom = wa < 0x8000u, ok = plain | in_rom | (wa - 0xFF00u < 4u);
                v = fast_load_u8(in_rom ? rom : memb, in_rom ? wa + (wa >> 14) * rom_off : off, ok, v);
                if (!ok) declined = true;
                if (wf & PDF_RD16) {  // POP / RET: the second byte, classified the same way
                    const uint32_t wb = (wa + 1) & 0xFFFF;
                    uint32_t off2;
                    const bool plain2 = fast_plain_offset(wb, off2), in_rom2 = wb < 0x8000u, ok2 = plain2 | in_rom2 | (wb - 0xFF00u < 4u);
                    v |= fast_load_u8(in_rom2 ? rom : memb, in_rom2 ? wb + (wb >> 14) * rom_off : off2, ok2, 0) << 8;
                    if (!ok2) declined = true;
                }
            }
        } else {  // single-lane build: branches are free (nothing diverges), the first matching region wins
            if (FAST && (wf & PDF_WR)) {
                wt = fast_store_target(wa);
                if (wt == FAST_WR_NONE) FAST_DECLINE();
                if ((mode & MODE_DEFER) && (wa - 0x8000u < 0x2000u || wa - 0xFE00u < 0x100u)) FAST_DECLINE();  // render_flush first
            }
            if (wf & PDF_RD) {
                v = rd8(wa);
                if (wf & PDF_RD16) v |= rd8((wa + 1) & 0xFFFF) << 8;
                if (FAST && declined) return false;
            }
        }
    }
    // ---- handler
    const uint32_t imm16 = d.y & 0xFFFFu, op = gb_prmt(d.x, 0, 0x4441), ex = gb_prmt(d.x, 0, 0x4442), f = hlaf >> 24;
    uint32_t rv = v, next_pc = d.y >> 16, wv = v, wn = wf & PDF_WR;
    cyc = d.x >> 24;
#define PAIR_OPERAND() (gb_prmt(bcde, hlaf, w >> 16) & 0xFFFFu)
    // SIMT: conditional / unconditional jumps are predicated, not dispatched (two selects on every lane), plain moves need no
    // handler at all, and INC / DEC and the ADD ADC SUB SBC CP group share ONE adder body (selects pick the operands): a warp
    // whose lanes run a mix of the four most frequent kinds of instruction takes a single path through here.
    // Single lane: one compare per kind, most frequent first, each with its own minimal body.
    const bool jump_taken = SIMT && (wf & PDF_JUMP) && ((f ^ ex) & op) == 0;
    if (SIMT) {
        next_pc = jump_taken ? imm16 : next_pc;
        cyc += jump_taken ? (ex & 0xF) : 0u;
    }
    if ((wf & PDF_MOV) || (SIMT && (wf & PDF_JUMP)) || (FAST && SIMT && declined)) {
        // rv = v
    } else if (!SIMT && (wf & PDF_JUMP)) {
        if (((f ^ ex) & op) == 0) { next_pc = imm16; cyc += ex & 0xF; }
    } else if (!SIMT && (wf & PDF_INCDEC)) {  // op = +1 / -1 (mod 256), ex = 0 / N|H: DEC inverts the half carry like a subtraction
        const uint32_t b = v & 0xFF, sum = b + op, res = sum & 0xFF;
        const uint32_t nf = (f & FLAG_C) | ((((b ^ op ^ sum) & 0x10) << 1) ^ ex) | (res == 0 ? FLAG_Z : 0);
        rv = res | (nf << 8);
        wv = res;
    } else if (wf & (PDF_INCDEC | PDF_ARITH)) {
        // a + x + cin with  INC / DEC: a = v, x = +1 / -1 (mod 256), no carry in, C kept, ex = 0 / N|H (DEC inverts the half carry
        // like a subtraction);  ADD..CP: a = A, x = v or its complement (ex = 0 / 0xFF), carry in for ADC / SBC (inverted for
        // the subtractions, whose H and C are the inverted carries)
        const bool inc = SIMT && (wf & PDF_INCDEC) != 0;
        const uint32_t b = v & 0xFF;
        const uint32_t a = inc ? b : ((hlaf >> 16) & 0xFF), x = inc ? op : (b ^ ex);
        const uint32_t cin = inc ? 0u : ((((f >> 4) & op) ^ ex) & 1);
        const uint32_t sum = a + x + cin, res = sum & 0xFF;
        const uint32_t hn = (((a ^ x ^ sum) & 0x10) << 1) ^ (ex & 0x60);
        const uint32_t cb = inc ? (f & FLAG_C) : (((sum >> 4) ^ ex) & 0x10);
        rv = res | ((hn | cb | (res == 0 ? FLAG_Z : 0)) << 8);
        wv = res;
    } else if (h == H_HLI) {
        rv = ((PAIR_OPERAND() + gb_prmt(d.x, 0, 0x9991)) & 0xFFFFu) | (v << 16);  // + sign-extended op
    } else switch (h) {
    case H_LOGIC: {  // AND: a & v; XOR: a ^ v; OR: (a & v) | (a ^ v)
        const uint32_t a = (hlaf >> 16) & 0xFF, b = v & 0xFF;
        const uint32_t res = ((a & b) & ex) | ((a ^ b) & op);
        rv = res | (((op ? 0 : FLAG_H) | (res == 0 ? FLAG_Z : 0)) << 8);
        break;
    }
    case H_ADD_HL: {
        const uint32_t hl = hlaf & 0xFFFF, ar = PAIR_OPERAND(), t = hl + ar;
        const uint32_t nf = (f & FLAG_Z) | (((hl & 0xFFF) + (ar & 0xFFF)) > 0xFFF ? FLAG_H : 0) | (t > 0xFFFF ? FLAG_C : 0);
        rv = (t & 0xFFFF) | (nf << 24);
        break;
    }
    case H_CALL: {
        if (((f ^ ex) & op) == 0) {  // high byte at SP-1 first, then low byte at SP-2
            if (FAST && !fast_stack_push(sp)) FAST_DECLINE();
            wa = (sp - 1) & 0xFFFF;
            if (FAST) wt = mem_offset(MEM_WRAM + (wa & 0x1FFF));
            wv = gb_prmt(next_pc, 0, 0x4401);
            wn = 2;
            sp = (sp - 2) & 0xFFFF;
            next_pc = imm16;
            cyc += ex & 0xF;
        }
        break;
    }
    case H_RET: {
        if (wf & PDF_RETI) m.ime = 1;
        if (((f ^ ex) & op) == 0) {
            next_pc = v & 0xFFFF;
            sp = (sp + 2) & 0xFFFF;
            cyc += ex & 0xF;
        }
        break;
    }
    case H_PUSH:
        if (FAST && !fast_stack_push(sp)) FAST_DECLINE();
        wa = (sp - 1) & 0xFFFF;
        if (FAST) wt = mem_offset(MEM_WRAM + (wa & 0x1FFF));
        wv = gb_prmt(PAIR_OPERAND(), 0, 0x4401);
        wn = 2;
        sp = (sp - 2) & 0xFFFF;
        break;
    case H_POP:
        rv = v & (0xFF00u | op);
        sp = (sp + 2) & 0xFFFF;
        break;
    case H_ROT: {  // branch-free: `ex` says where the shifted-in bit comes from (pd_rot_ex)
        const uint32_t b = v & 0xFF, c = (f >> 4) & 1, right = ex & 1, b7 = b >> 7;
        uint32_t cout = right ? (b & 1) : b7;
        const uint32_t in = (((ex >> 1) & cout) | ((ex >> 2) & c) | ((ex >> 3) & b7)) & 1;
        uint32_t res = right ? ((b >> 1) | (in << 7)) : (((b << 1) | in) & 0xFF);
        if (ex & 0x10) { res = ((b >> 4) | (b << 4)) & 0xFF; cout = 0; }  // SWAP
        const uint32_t nf = ((res == 0 && !(op & 8)) ? FLAG_Z : 0) | (cout << 4);  // RLCA..RRA clear Z
        rv = res | (nf << 8);
        wv = res;
        break;
    }
    case H_CPL: rv = (~(hlaf >> 16) & 0xFF) | ((f | FLAG_N | FLAG_H) << 8); break;
    case H_IME: m.ime = op; break;
    case H_JPHL: next_pc = hlaf & 0xFFFF; break;
    case H_BIT: rv = ((f & FLAG_C) | FLAG_H | ((v & imm16 & 0xFF) ? 0 : FLAG_Z)) << 8; break;
    case H_RESSET:
        rv = (v & imm16 & 0xFF) | (imm16 >> 8);
        wv = rv;
        break;
    default: {  // H_RARE / H_SLOW (never in the fast body): `op` is the opcode
        if (FAST) {
            FAST_DECLINE();
            break;
        }
        const uint32_t a = (hlaf >> 16) & 0xFF, hl = hlaf & 0xFFFF;
        switch (op) {
        case 0x76: m.halted = 1; mode |= MODE_ATTN | MODE_POST; next_pc = r.pc; break;  // HALT: PC stays on the HALT byte
        case 0x10: break;                                                                // STOP skips a byte
        case 0xF3: m.ime = 0; break;
        case 0xFB: m.ime = 1; break;  // PyBoy: EI takes effect immediately
        case 0x27: {                  // DAA
            uint32_t corr = ((f & FLAG_H) ? 0x06 : 0) | ((f & FLAG_C) ? 0x60 : 0), t = a;
            if (f & FLAG_N) {
                t -= corr;
            } else {
                if ((t & 0x0F) > 9) corr |= 0x06;
                if (t > 0x99) corr |= 0x60;
                t += corr;
            }
            t &= 0xFF;
            hlaf = (hlaf & 0xFFFF) | (t << 16) | (((f & FLAG_N) | (t == 0 ? FLAG_Z : 0) | ((corr & 0x60) ? FLAG_C : 0)) << 24);
            break;
        }
        case 0x2F: hlaf = (hlaf & 0xFFFF) | ((~a & 0xFF) << 16) | ((f | FLAG_N | FLAG_H) << 24); break;    // CPL
        case 0x37: hlaf = (hlaf & 0x00FFFFFFu) | (((f & FLAG_Z) | FLAG_C) << 24); break;                   // SCF
        case 0x3F: hlaf = (hlaf & 0x00FFFFFFu) | (((f & FLAG_Z) | ((f & FLAG_C) ^ FLAG_C)) << 24); break;  // CCF
        case 0x08: wa = imm16; wv = sp; wn = 3; break;                                                    // LD (nn),SP
        case 0xE8:
        case 0xF8: {  // ADD SP,e / LD HL,SP+e
            const uint32_t imm8 = imm16 & 0xFF;
            const uint32_t nf = (((sp & 0xF) + (imm8 & 0xF)) > 0xF ? FLAG_H : 0) | (((sp & 0xFF) + imm8) > 0xFF ? FLAG_C : 0);
            const uint32_t t = (sp + ((imm8 ^ 0x80) - 0x80)) & 0xFFFF;
            hlaf = (hlaf & 0x00FFFFFFu) | (nf << 24);
            if (op == 0xE8) sp = t;
            else hlaf = (hlaf & 0xFFFF0000u) | t;
            break;
        }
        case 0xE9: next_pc = hl; break;                 // JP HL
        case 0xF9: sp = hl; break;                      // LD SP,HL
        case 0x31: sp = imm16; break;                   // LD SP,nn
        case 0x33: sp = (sp + 1) & 0xFFFF; break;       // INC SP
        case 0x3B: sp = (sp + 0xFFFF) & 0xFFFF; break;  // DEC SP
        case 0x39: {                                    // ADD HL,SP
            const uint32_t t = hl + sp;
            const uint32_t nf = (f & FLAG_Z) | (((hl & 0xFFF) + (sp & 0xFFF)) > 0xFFF ? FLAG_H : 0) | (t > 0xFFFF ? FLAG_C : 0);
            hlaf = (hlaf & 0x00FF0000u) | (t & 0xFFFF) | (nf << 24);
            break;
        }
        case 0xE2: wa = 0xFF00u | (bcde & 0xFF); wv = a; wn = PDF_WR; break;                                      // LD (FF00+C),A
        case 0xF2: hlaf = (hlaf & 0xFF00FFFFu) | (bus_read_full(m, 0xFF00u | (bcde & 0xFF)) << 16); break;        // LD A,(FF00+C)
        default: m.fault = 1; break;  // illegal opcode: PyBoy raises; 1-byte 4-cycle NOP + sticky fault
        }
        break;
    }
    }
#undef PAIR_OPERAND
#if !defined(GB_HOSTSIM) && !defined(GB_OPT_NO_JOIN)
    if (FAST && SIMT) {
        // Opaque join: the empty asm keeps nvcc from threading the handlers that cannot decline straight to the write-back,
        // past this test.  With every path through here, this point post-dominates the handler dispatch and gets a
        // re-convergence barrier (BSYNC): the write-back, the stores and the loop tail run once per warp.
        uint32_t dj = declined;
        asm volatile("" : "+r"(dj));
        declined = dj != 0;
    }
#endif
    if (FAST && declined) return false;  // nothing has been changed
#undef FAST_DECLINE
    // ---- register write-back (uniform)
    r.bcde = gb_prmt(bcde, rv, d.z);
    r.hlaf = gb_prmt(hlaf, rv, d.z >> 16);
    r.sp = sp;
    r.pc = next_pc;
    // ---- bus writes.  wn = PDF_WR: byte wv at wa; 2: low byte of wv at wa, then high byte at wa - 1 (pushes); 3: low byte
    // at wa, then high byte at wa + 1 (LD (nn),SP)
    if (wn) {
        if (FAST) {
            if (wt < FAST_WR_P1) {  // plain RAM; a push (both bytes in work RAM, checked by the handler) adds its high byte below
                memb[wt] = (uint8_t)wv;
                if (wn == 2) memb[mem_offset(MEM_WRAM + ((wa - 1) & 0x1FFF))] = (uint8_t)(wv >> 8);
            } else if (wt == FAST_WR_P1) {  // joypad matrix select (a game's input routine writes it several times a frame)
                memb[mem_offset(MEM_HI + 0x100)] = (uint8_t)joypad_pull(m, wv & 0xFF);
            } else if (wt == FAST_WR_BANK) {  // MBC3 ROM bank select (constant traffic in banked games)
                uint32_t bank = wv & 0x7F;
                bank = bank ? bank : 1;
                m.rombank = bank;
                rom_off = (bank_mask ? (bank & bank_mask) : (bank % m.rom_banks)) * 0x4000u - 0x4000u;
                m.rom_off = rom_off;
            }
        } else {
            const uint32_t count = (wn & 3) ? 2u : 1u, second = (wn == 2 ? wa - 1 : wa + 1) & 0xFFFF;
            for (uint32_t i = 0; i < count; i++) bus_write_full(m, i ? second : wa, (i ? wv >> 8 : wv) & 0xFF);
        }
    }
    return true;
}

// Single-lane build: dispatch on the class id of the control word to an instance of the body in which handler and operand
// flags are constants.  This replaces the ~10 flag tests + branches the generic body spends per instruction (12.3 BRA and
// 17.7 LOP3 of its 68 SASS instructions per emulated one); nothing diverges in a single-thread block, so the code-size price
// (34 short bodies) is the only one.  nvcc lowers a switch to a balanced compare tree (five tests for every class, hot or
// cold), so the dispatch is the tree gb_classes.inc spells out as explicit tests, shaped by the class mix of the benchmark
// workloads (tools/class_mix.py): the hottest class takes two tests, 3.6 per instruction on average.  Each test sees
// the class id through an empty asm, so that nvcc cannot merge the tests back into a switch.
__device__ __forceinline__ void gb_opaque(uint32_t &v) {  // the compiler no longer knows v's value (it is unchanged)
#if !defined(GB_HOSTSIM)
    asm volatile("" : "+r"(v));
#endif
}
__device__ __forceinline__ bool cpu_exec_by_class(Machine &m, const uint4 d, CpuRegs &r, uint32_t &rom_off, uint32_t &mode, uint32_t &cyc, uint8_t *memb,
                                                  const uint8_t *rom, uint32_t bank_mask) {
    uint32_t c = PD_CLASS(d.w);
#define GB_CLS_TEST(t) (gb_opaque(c), (t))
#define GB_CLS_RUN(id, H, F) return cpu_exec<true, false, H, F>(m, d, r, rom_off, mode, cyc, memb, rom, bank_mask);
    GB_CLS_DISPATCH(c, GB_CLS_RUN, return false;)  // rare opcodes, on-the-fly decode: the slow tick
#undef GB_CLS_RUN
#undef GB_CLS_TEST
}

// The fast body of the lock-step build (k_run_frames, several envs per warp) as ONE straight line of code: no handler
// dispatch at all.  Every lane computes the result of every kind of instruction the fast set knows -- the adder, the logic
// unit, the rotator, BIT / RES / SET, CPL, the 16-bit increments and ADD HL, POP's mask, the branch condition -- from its own
// control word, and selects pick what is written back; loads and stores are predicated.  A warp whose lanes are at
// different instructions (the normal state of affairs: its envs are at different places of the game) therefore issues the
// same instruction stream as a warp in lock-step; what it costs is the longest dependency chain (descriptor -> operand ->
// ALU -> write-back), not the sum of the handlers its lanes happen to need.  Returns false, having changed nothing, for
// whatever is outside the fast set (cpu_tick_slow redoes the tick).
__device__ __forceinline__ bool cpu_exec_lockstep(Machine &m, const uint4 d, CpuRegs &r, uint32_t &rom_off, uint32_t mode, uint32_t &cyc, uint8_t *memb,
                                                  const uint8_t *rom, uint32_t bank_mask, bool declined) {
    const uint32_t bcde = r.bcde, hlaf = r.hlaf, sp = r.sp;
    const uint32_t w = d.w, h = d.x & 0xFF, op = gb_prmt(d.x, 0, 0x4441), ex = gb_prmt(d.x, 0, 0x4442), imm16 = d.y & 0xFFFFu, fall = d.y >> 16;
    const uint32_t f = hlaf >> 24, a8 = (hlaf >> 16) & 0xFF, hl = hlaf & 0xFFFF;
    declined |= h >= H_RARE;
    // ---- control: the branch condition (mask in op, expected flag value in ex; unconditional: mask 0)
    const bool cond = ((f ^ ex) & op) == 0;
    const bool is_call = h == H_CALL, is_ret = h == H_RET, is_push = h == H_PUSH, is_pop = h == H_POP;
    const bool jumps = cond && ((w & PDF_JUMP) || is_call), returns = cond && is_ret, pushes = (cond && is_call) || is_push;
    // ---- operand and address
    uint32_t v = gb_prmt(bcde, hlaf, w);  // byte 0 = source register
    v = (w & PDF_IMM) ? imm16 : v;
    const uint32_t pair = gb_prmt(bcde, hlaf, w >> 16) & 0xFFFFu;
    uint32_t wa = (w & PDF_AIMM) ? imm16 : pair;
    wa = (w & PDF_ASP) ? sp : wa;
    wa = pushes ? ((sp - 1) & 0xFFFF) : wa;
    uint32_t off;
    const bool plain = fast_plain_offset(wa, off);
    const bool rd = (w & PDF_RD) != 0, rd16 = (w & PDF_RD16) != 0, wr = (w & PDF_WR) != 0;
    // stores outside plain RAM: MBC3 bank select, sound registers (dropped), P1; anything else is not for the fast body
    const bool wr_special = wr && !plain;
    const uint32_t wt = (wa - 0x2000u < 0x2000u) ? FAST_WR_BANK : (wa - 0xFF10u < 0x30u) ? FAST_WR_DROP : wa == 0xFF00u ? FAST_WR_P1 : FAST_WR_NONE;
    declined |= wr_special && wt == FAST_WR_NONE;
    declined |= pushes && !fast_stack_push(sp);
    declined |= wr && (mode & MODE_DEFER) && (wa - 0x8000u < 0x2000u || wa - 0xFE00u < 0x100u);  // deferred PPU: render_flush first
    // loads: first byte from plain RAM, ROM or P1 / SB / SC; the second byte of POP / RET (always at SP + 1) from work RAM
    const bool in_rom = wa < 0x8000u, rd_ok = plain || in_rom || (wa - 0xFF00u < 4u), rd16_ok = sp - 0xC000u < 0x3DFFu;
    declined |= (rd && !rd_ok) || (rd16 && !rd16_ok);
    v = fast_load_u8(in_rom ? rom : memb, in_rom ? wa + (wa >> 14) * rom_off : off, rd && rd_ok, v);
    v |= fast_load_u8(memb, mem_offset(MEM_WRAM + ((sp + 1) & 0x1FFF)), rd16 && rd16_ok, 0) << 8;
    const uint32_t b = v & 0xFF, b7 = b >> 7;
    // ---- every unit computes
    // adder.  INC / DEC: a = v, x = +1 / -1, C kept, ex = 0 / N|H;  ADD ADC SUB SBC CP: a = A, x = v or its complement (ex = 0 / 0xFF)
    const bool inc = (w & PDF_INCDEC) != 0;
    const uint32_t ad_a = inc ? b : a8, ad_x = inc ? op : (b ^ ex), ad_c = inc ? 0u : ((((f >> 4) & op) ^ ex) & 1);
    const uint32_t sum = ad_a + ad_x + ad_c, ad_res = sum & 0xFF;
    const uint32_t ad_f = ((((ad_a ^ ad_x ^ sum) & 0x10) << 1) ^ (ex & 0x60)) | (inc ? (f & FLAG_C) : (((sum >> 4) ^ ex) & 0x10)) | (ad_res == 0 ? FLAG_Z : 0);
    // logic: AND a & v; XOR a ^ v; OR (a & v) | (a ^ v)
    const uint32_t lg_res = ((a8 & b) & ex) | ((a8 ^ b) & op);
    const uint32_t lg_f = (op ? 0 : FLAG_H) | (lg_res == 0 ? FLAG_Z : 0);
    // rotates and shifts (pd_rot_ex)
    const uint32_t right = ex & 1;
    uint32_t rt_c = right ? (b & 1) : b7;
    const uint32_t rt_in = (((ex >> 1) & rt_c) | ((ex >> 2) & (f >> 4)) | ((ex >> 3) & b7)) & 1;
    uint32_t rt_res = right ? ((b >> 1) | (rt_in << 7)) : (((b << 1) | rt_in) & 0xFF);
    rt_res = (ex & 0x10) ? (((b >> 4) | (b << 4)) & 0xFF) : rt_res;
    rt_c = (ex & 0x10) ? 0u : rt_c;
    const uint32_t rt_f = ((rt_res == 0 && !(op & 8)) ? FLAG_Z : 0) | (rt_c << 4);
    // 16-bit: INC rr / DEC rr / HL+ / HL- and ADD HL,rr
    const uint32_t hli = ((pair + gb_prmt(d.x, 0, 0x9991)) & 0xFFFFu) | (v << 16);
    const uint32_t t16 = hl + pair;
    const uint32_t addhl = (t16 & 0xFFFF) | (((f & FLAG_Z) | (((hl & 0xFFF) + (pair & 0xFFF)) > 0xFFF ? FLAG_H : 0) | (t16 > 0xFFFF ? FLAG_C : 0)) << 24);
    // ---- select the result: 8-bit results travel as res | new F << 8 (the write-back selectors say what is kept)
    uint32_t rv = v;
    rv = (w & (PDF_INCDEC | PDF_ARITH)) ? (ad_res | (ad_f << 8)) : rv;
    rv = h == H_LOGIC ? (lg_res | (lg_f << 8)) : rv;
    rv = h == H_ROT ? (rt_res | (rt_f << 8)) : rv;
    rv = h == H_BIT ? (((f & FLAG_C) | FLAG_H | ((b & imm16) ? 0 : FLAG_Z)) << 8) : rv;
    rv = h == H_RESSET ? ((b & imm16) | (imm16 >> 8)) : rv;
    rv = h == H_CPL ? ((~a8 & 0xFF) | ((f | FLAG_N | FLAG_H) << 8)) : rv;
    rv = h == H_HLI ? hli : rv;
    rv = h == H_ADD_HL ? addhl : rv;
    rv = is_pop ? (v & (0xFF00u | op)) : rv;
    // ---- next PC, stack pointer, cycles
    uint32_t next_pc = jumps ? imm16 : fall;
    next_pc = returns ? (v & 0xFFFF) : next_pc;
    next_pc = h == H_JPHL ? hl : next_pc;
    cyc = (d.x >> 24) + ((jumps || returns) ? (ex & 0xF) : 0u);
    const uint32_t new_sp = (sp + ((is_pop || returns) ? 2u : 0u) - (pushes ? 2u : 0u)) & 0xFFFF;
    // ---- what a store writes: the unit's 8-bit result (the register itself for LD (HL+-),A); a push the pair or the return
    // address, high byte first
    uint32_t wv = h == H_HLI ? v : rv;
    wv = pushes ? gb_prmt(is_push ? pair : fall, 0, 0x4401) : wv;
    if (declined) return false;  // nothing has been changed
    r.bcde = gb_prmt(bcde, rv, d.z);
    r.hlaf = gb_prmt(hlaf, rv, d.z >> 16);
    r.sp = new_sp;
    r.pc = next_pc;
    if ((wr && plain) || pushes) memb[off] = (uint8_t)wv;
    if (pushes) memb[mem_offset(MEM_WRAM + ((sp - 2) & 0x1FFF))] = (uint8_t)(wv >> 8);
    if (wr_special) {
        if (wt == FAST_WR_P1) {  // joypad matrix select (a game's input routine writes it several times a frame)
            memb[mem_offset(MEM_HI + 0x100)] = (uint8_t)joypad_pull(m, wv & 0xFF);
        } else if (wt == FAST_WR_BANK) {  // MBC3 ROM bank select (constant traffic in banked games)
            uint32_t bank = wv & 0x7F;
            bank = bank ? bank : 1;
            m.rombank = bank;
            rom_off = (bank_mask ? (bank & bank_mask) : (bank % m.rom_banks)) * 0x4000u - 0x4000u;
            m.rom_off = rom_off;
        }
    }
    if ((w & PDF_RETI) || h == H_IME) m.ime = h == H_IME ? op : 1u;
    return true;
}

// One whole tick on the parked machine, for everything the fast loop declines: CPU.tick (interrupt check, HALT, one
// instruction from anywhere, through the full bus) followed by Motherboard.tick's HALT fast-forward and Timer.tick's TIMA
// half.  The caller has brought the clocks up to date; returns the T-cycles to advance them by.
// While TIMA runs and the CPU is not halted the caller accounts the returned cycles to the TIMA counter lazily (time_sync);
// a halted tick advances the timer here, by its fast-forwarded cycle count, and says so in `timer_ticked`.
__device__ GB_NOINLINE uint32_t cpu_tick_slow(Machine &m, const uint4 *__restrict__ rom_dec, uint32_t bank_mask, uint32_t &timer_ticked) {
    uint32_t cyc = 0;
    bool execute = true;
    if (m.halted | m.iq | (m.iflag & m.ie & 0x1F)) {
        const uint32_t r = cpu_attention(m);
        execute = r & 1;
        cyc = r >> 8;
    }
    if (execute) {
        const uint32_t pc = m.pc;
        uint4 d = make_uint4(H_SLOW, 0, 0, PD_NO_CLASS_W);
        if (pc < 0x8000u) d = __ldg(rom_dec + (pc + (pc >> 14) * m.rom_off));
        if ((d.x & 0xFF) == H_SLOW) d = cpu_decode_slow(m, pc);
        CpuRegs r = {m.bcde, m.hlaf, m.sp, pc};
        uint32_t rom_off = m.rom_off, mode = 0;
        cpu_exec<false, false>(m, d, r, rom_off, mode, cyc, m.memb, m.rom, bank_mask);
        m.bcde = r.bcde; m.hlaf = r.hlaf; m.sp = r.sp; m.pc = r.pc;
        m.n_instr++;
    }
    timer_ticked = m.halted;
    if (m.halted) cyc = cpu_post_slow(m, cyc);
    return cyc;
}

// HRAM-resident code (every game keeps its OAM-DMA stub there, ~80 instructions per frame): decoded inline from two
// aligned words, no bus, no call
__device__ __forceinline__ uint4 cpu_decode_hram(const uint8_t *memb, uint32_t pc) {
    const uint32_t i = MEM_HI + (pc - 0xFE00), sh = (i & 3) * 8;
    const uint32_t w0 = ((const uint32_t *)memb)[(i >> 2) << 5], w1 = ((const uint32_t *)memb)[((i >> 2) + 1) << 5];
    const uint32_t ins = sh ? ((w0 >> sh) | (w1 << (32 - sh))) : w0;
    return pd_finish(c_base_desc[(ins & 0xFF) == 0xCB ? (256u | ((ins >> 8) & 0xFF)) : (ins & 0xFF)], ins, pc);
}

// The fast loop: no call inside (a call in this loop makes the compiler save convergence-barrier state to the stack on
// every iteration).  Returns true when the countdown has reached the deadline, false when an instruction needs the slow tick.
// CLASSES (single-lane build only): dispatch on the class id of the control word (cpu_exec_by_class).
template <bool SIMT, bool CLASSES>
__device__ __forceinline__ bool cpu_fast_loop(Machine &m, const RunCtx &cx, CpuRegs &r, uint32_t &rom_off, uint32_t &mode, uint32_t &n_instr, int &rem,
                                              uint8_t *memb, const uint8_t *rom) {
    for (;;) {
        uint32_t cyc;
        // ONE instance of the instruction body: the descriptor comes from the pre-decoded ROM table or, for the HRAM stub,
        // from an inline decode -- lanes running either kind of code meet again in front of cpu_exec.  SIMT: a lane that
        // has to leave the loop (interrupt pending, HALT, code in other RAM) goes through the body as `declined`.
        uint4 d = make_uint4(H_SLOW, 0, 0x32103210u, PD_NO_CLASS_W);
        bool leave = false;
        const uint32_t pc = r.pc;
        if (!((pc | mode) & (0x8000u | MODE_POST))) {  // ROM code, nothing pending, not halted
            d = __ldg(cx.rom_dec + (pc + (pc >> 14) * rom_off));
        } else if (!(mode & (MODE_ATTN | MODE_POST)) && pc - 0xFF80u < 0x7Du) {
            d = cpu_decode_hram(memb, pc);
        } else {
            if (!SIMT) return false;
            leave = true;
        }
        if (SIMT) {
#if !defined(GB_OPT_LOCKSTEP)  // the fully predicated body lost on B200 (400 k vs 620 k env-steps/s at 32,768 envs): see cpu_exec_lockstep
            if (!cpu_exec<true, true>(m, d, r, rom_off, mode, cyc, memb, rom, cx.bank_mask, leave)) return false;
#else
            if (!cpu_exec_lockstep(m, d, r, rom_off, mode, cyc, memb, rom, cx.bank_mask, leave)) return false;
#endif
        } else if (CLASSES) {
            if (!cpu_exec_by_class(m, d, r, rom_off, mode, cyc, memb, rom, cx.bank_mask)) return false;
        } else {
            if (!cpu_exec<true, false>(m, d, r, rom_off, mode, cyc, memb, rom, cx.bank_mask, leave)) return false;
        }
        GB_TRACE_SLOT(0, pc < 0x8000u ? pc + (pc >> 14) * rom_off : (0xF00000u | pc), d.x, d.w);
        n_instr++;
        rem -= (int)cyc;
        if (rem <= 0) return true;
    }
}

// Interprets until this env's LCD clock reaches its next hard event (lcd_deadline).  `m` is the env's machine in shared
// memory; the SM83 registers, the ROM bank offset, the cycle countdown and the mode word are cached in registers.
template <bool SIMT>
__device__ __forceinline__ void cpu_run_to_event(Machine &m, const RunCtx &cx) {
    CpuRegs r = {m.bcde, m.hlaf, m.sp, m.pc};
    uint32_t rom_off = m.rom_off, n_instr = m.n_instr;
    uint8_t *memb = m.memb;
    const uint8_t *rom = m.rom;
    int rem = hot_rem(m, true);
    m.t_sync = rem;
    uint32_t mode = hot_mode(m), timer_pending = 0;
again:
    do {
        // ---- fast loop (cpu_fast_loop).  The single-lane build has two copies: class-dispatched bodies (34 of them: a large
        // hot set that pays when the loop runs long) and, while TIMA runs -- the countdown then ends every few instructions and
        // the loop's entry / exit paths are as hot as its body -- the compact generic one.
        bool at_deadline;
        if (!SIMT && !(m.tmr & TIMA_ON)) at_deadline = cpu_fast_loop<SIMT, true>(m, cx, r, rom_off, mode, n_instr, rem, memb, rom);
        else at_deadline = cpu_fast_loop<SIMT, false>(m, cx, r, rom_off, mode, n_instr, rem, memb, rom);
        if (at_deadline) {
            timer_pending = 1;
            goto deadline;
        }
        {
            // ---- slow tick.  Park the registers, bring the clocks up to date, apply the soft LCD events that have become due
            // (never a hard one: the loop stops at those) -- the machine in shared memory is now exactly PyBoy's at this
            // instruction boundary -- and run the tick out of line.  Nothing hot is live across the call.
            m.bcde = r.bcde; m.hlaf = r.hlaf; m.sp = r.sp; m.pc = r.pc; m.n_instr = n_instr;
            time_sync(m, rem);
            if (m.lazy && (int)(m.clock - m.target) >= 0) lcd_catch_up(m);
            GB_TRACE_SLOT(1, m.pc < 0x8000u ? m.pc + (m.pc >> 14) * m.rom_off : (0xF00000u | m.pc), 0, 0);
            uint32_t timer_ticked;
            const uint32_t cyc = cpu_tick_slow(m, cx.rom_dec, cx.bank_mask, timer_ticked);
            r.bcde = m.bcde; r.hlaf = m.hlaf; r.sp = m.sp; r.pc = m.pc; n_instr = m.n_instr; rom_off = m.rom_off;
            memb = m.memb; rom = m.rom;
            // the tick's cycles reach clock / DIV / TIMA counter at the next time_sync; a halted tick has advanced the TIMA
            // counter already: take them out again (modulo 2^32; the counter is only compared when it is in sync)
            if (timer_ticked && (m.tmr & TIMA_ON)) m.timac -= cyc;
            timer_pending = !timer_ticked;
            rem = hot_rem(m, false);  // the tick may have changed what the countdown and the mode word derive from
            m.t_sync = rem;
            mode = hot_mode(m);
            rem -= (int)cyc;
        }
    } while (rem > 0);
deadline:
    m.bcde = r.bcde; m.hlaf = r.hlaf; m.sp = r.sp; m.pc = r.pc; m.n_instr = n_instr;
    time_sync(m, rem);
    if (timer_pending) timer_tick_tima(m, 0);  // Timer.tick's TIMA half of the tick that ended here, unless a halted tick did it itself
    if ((m.tmr & TIMA_ON) && !m.halted) {
        // a running TIMA ends the countdown at every increment (every 16 cycles at the fastest rate): unless the LCD is due as
        // well, re-arm the countdown and carry on instead of going back through the frame loop
        const bool lcd_due = (m.lcdc & 0x80) ? (int)(m.clock - m.target) >= 0 : m.clock >= FRAME_CYCLES;
        if (!lcd_due) {
            rem = hot_rem(m, true);
            m.t_sync = rem;
            mode = hot_mode(m);
            timer_pending = 0;
            if (rem > 0) goto again;
        }
    }
}
