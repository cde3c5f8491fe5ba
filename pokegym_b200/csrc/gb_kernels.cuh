// gb_kernels.cuh -- emulation kernels: the 24-frame step, state scatter/gather, bus access.
#pragma once
#include "gb_cpu.cuh"
#include "gb_device.cuh"

// 64-thread blocks, 12 of them per SM: an 80-register budget (at 64 registers the loop-entry paths spill the machine pointer and
// the barrier state: 610 k vs 629 k env-steps/s at 32,768 envs) and 24 resident warps per SM -- the lanes policy (gbenv.cu) never
// asks for more than 16 per SM below 113k envs.
#define STEP_THREADS 64
#define STEP_MIN_BLOCKS 12

// pyboy_binding.ACTIONS (:40) Down Left Right Up A B Start Select -> joypad button ids
// (Right Left Up Down A B Select Start, the bit order of PyBoy's Interaction nibbles)
__constant__ int c_action_button[8] = {3, 1, 0, 2, 4, 5, 7, 6};

struct RunParams {
    DevArrays d;
    const uint8_t *actions;  // may be null: plain ticks without input
    const uint8_t *skip;     // may be null; envs with skip[e] != 0 are not run (gbenv_step_masked)
    int n_frames;
    int render_mode;  // 0: renderer disabled, 1: enabled on every frame, 2: enabled on the last frame only
    int release_frame;  // frame index at which the button is released (8 in the reference)
    int lanes;          // envs per warp (1..32): fewer lanes = more warps = more latency hiding
    int defer;          // deferred PPU: record the lines of the rendered frame (d.dl), k_render_pending draws them
    uint32_t bank_mask;  // rom_banks - 1 when the bank count is a power of two, else 0
    unsigned long long *counters;  // [0] instructions, [1] cycles, [2] frames, [3] faults
};

// Per-env slot in shared memory: the machine.
// The slot stride is an odd number of 8-byte units, so the same field of 32 consecutive slots falls into 16 banks
// (two-way conflicts, on cold paths only: the hot state is in registers).  The renderer's line buffer and sprite sort
// keys follow as [word][slot] arrays (conflict-free).
struct EnvSlot {
    Machine m;
};
#define ENV_SLOT_STRIDE ((sizeof(EnvSlot) + 7) / 8 * 8 + ((((sizeof(EnvSlot) + 7) / 8) & 1) ? 0 : 8))
#define ENV_SMEM_BYTES(nslots) ((size_t)(nslots) * (ENV_SLOT_STRIDE + (FB_LINE_WORDS + 10) * 4))

// The frame loop of one env (pyboy_binding.run_action_on_emulator :71-91 around Motherboard.tick).  It is organised
// around LCD events: cpu_run_to_event interprets until this env's LCD clock reaches its next mode change, then the
// mode change is performed (scanline parameters, rendering, LY/STAT/interrupt flags).  All envs see the same number
// of LCD events per frame, so a warp re-converges 442 times a frame and the scanline renderer runs with every lane.
template <bool SIMT>
__device__ __forceinline__ void run_frames_env(Machine &m, const RunParams &p, int button) {
    RunCtx cx;
    cx.rom_dec = p.d.rom_dec;
    cx.bank_mask = p.bank_mask;
    for (int frame = 0; frame < p.n_frames; frame++) {
        if (m.defer_from != m.defer_next) render_flush(m);  // deferred lines of the frame before (every frame is rendered: tick)
        // PyBoy.tick applies queued inputs before Motherboard.tick
        if (button >= 0) {
            if (frame == 0) joypad_event(m, button, 1);
            if (frame == p.release_frame) joypad_event(m, button, 0);
        }
        m.disable_renderer = p.render_mode == 1 ? 0 : p.render_mode == 2 ? (frame != p.n_frames - 1) : 1;
        // Motherboard.tick: while lcd.processing_frame()
        bool done = m.frame_done;
        m.frame_done = 0;
        while (!done) {
            GB_TRACE_SLOT(2, 0, 0, 0);  // the lanes of a warp re-converge here
            if (m.halted && !(m.iq | (m.iflag & m.ie & 0x1F) | (m.tmr & 0x04000000u)) && (m.lcdc & 0x80)) {
                // Quiet HALT (nothing pending, TIMA stopped): CPU.tick is a no-op and Motherboard.tick jumps from LCD mode
                // change to mode change; only a hard one (VBlank entry, a rendered HBlank) can end the HALT or the frame,
                // so jump there without entering the interpreter.
                const int a = lcd_deadline(m);
                if (a > 0) { m.divc += a; m.clock += a; }
            } else {
                cpu_run_to_event<SIMT>(m, cx);
            }
            lcd_catch_up(m);
            done = m.frame_done;
            m.frame_done = 0;
        }
    }
}

// One thread per env; `lanes` envs per warp (the first `lanes` threads of each warp carry one; 32 = a full tile per
// warp).  Runs `n_frames` whole frames without returning to the host.
#if !defined(GB_HOSTSIM)
extern __shared__ unsigned long long s_env_slots[];
__global__ void __launch_bounds__(STEP_THREADS, STEP_MIN_BLOCKS) k_run_frames(RunParams p) {
    const int tid = threadIdx.x;
    const int warp = (blockIdx.x * STEP_THREADS + tid) >> 5, wl = tid & 31;
    if (wl >= p.lanes) return;  // partial-warp mode: only the first `lanes` threads of each warp carry an env
    const int env = warp * p.lanes + wl;
    if (env >= p.d.n_envs || (p.skip && p.skip[env])) return;
    const int tile = env >> 5, lane = env & 31;
    const uint32_t nslots = (STEP_THREADS / 32) * p.lanes, si = (tid >> 5) * p.lanes + wl;
    EnvSlot &slot = *(EnvSlot *)((char *)s_env_slots + (size_t)si * ENV_SLOT_STRIDE);
    uint32_t *const line = (uint32_t *)((char *)s_env_slots + (size_t)nslots * ENV_SLOT_STRIDE) + si, *const keys = line + FB_LINE_WORDS * nslots;
    Machine &m = slot.m;
    machine_load(m, p.d, tile, lane);
    m.rline = line; m.rkeys = keys; m.rls = nslots;
    if (p.defer && p.d.dl) m.dl = p.d.dl + il_index(tile, DL_WORDS, 0, lane);
    const int button = p.actions ? c_action_button[p.actions[env] & 7] : -1;
    run_frames_env<true>(m, p, button);
    machine_store(m, p.d, tile, lane);
    if (p.counters) {
        atomicAdd(&p.counters[0], (unsigned long long)m.n_instr);
        atomicAdd(&p.counters[1], (unsigned long long)m.n_cycles);
        atomicAdd(&p.counters[2], (unsigned long long)p.n_frames);
    }
}

// The same with ONE THREAD PER BLOCK, for batches small enough that every env gets a warp of its own anyway (lanes == 1:
// up to 32 blocks x 148 SMs = 4,736 envs in one wave).  With __launch_bounds__(1) ptxas knows that no branch can diverge and
// emits none of the convergence-barrier scaffolding (BSSY / BSYNC / BREAK / BMOV: about one instruction in nine of the
// multi-lane build's hot loop), keeps loop-invariant addresses in uniform registers and needs no spills.
#define STEP1_MIN_BLOCKS 32
__global__ void __launch_bounds__(1, STEP1_MIN_BLOCKS) k_run_frames_1(RunParams p) {
    const int env = blockIdx.x;
    if (env >= p.d.n_envs || (p.skip && p.skip[env])) return;
    const int tile = env >> 5, lane = env & 31;
    EnvSlot &slot = *(EnvSlot *)((char *)s_env_slots);
    uint32_t *const line = (uint32_t *)((char *)s_env_slots + ENV_SLOT_STRIDE), *const keys = line + FB_LINE_WORDS;
    Machine &m = slot.m;
    machine_load(m, p.d, tile, lane);
    m.rline = line; m.rkeys = keys; m.rls = 1;
    if (p.defer && p.d.dl) m.dl = p.d.dl + il_index(tile, DL_WORDS, 0, lane);
    const int button = p.actions ? c_action_button[p.actions[env] & 7] : -1;
    run_frames_env<false>(m, p, button);
    machine_store(m, p.d, tile, lane);
    if (p.counters) {
        atomicAdd(&p.counters[0], (unsigned long long)m.n_instr);
        atomicAdd(&p.counters[1], (unsigned long long)m.n_cycles);
        atomicAdd(&p.counters[2], (unsigned long long)p.n_frames);
    }
}
#endif

// Deferred PPU, second half: draws the lines an env's emulation left recorded (R_MISC: [defer_from, defer_next)).
// `y0`, `dy`: this caller's share of the lines (the kernel: one line per thread; the host harness: all of them).  Returns whether the
// env had pending lines.
__device__ __forceinline__ bool render_pending_lines(const DevArrays &d, int tile, int lane, uint32_t y0, uint32_t dy, uint32_t *line, uint32_t *keys, uint32_t ls) {
    const uint32_t misc = d.regs[il_index(tile, R_WORDS, R_MISC, lane)], from = (misc >> 8) & 0xFF, next = (misc >> 16) & 0xFF;
    if (from >= next) return false;
    Machine r;
    machine_bind(r, d, tile, lane);
    const uint32_t *dl = d.dl + il_index(tile, DL_WORDS, 0, lane);
    for (uint32_t y = y0; y < next; y += dy) {
        if (y < from) continue;
        const uint32_t w0 = dl[(y * 3 + 0) << 5], w1 = dl[(y * 3 + 1) << 5], w2 = dl[(y * 3 + 2) << 5];
        r.scroll = w0; r.lcdc = w1 & 0xFF; r.pal = w1 >> 8; r.ly_window = (int)w2;
        render_line(r, y, line, keys, ls);
    }
    return true;
}

#if !defined(GB_HOSTSIM)
// grid (tiles, 144 / RENDER_LINES_PER_BLOCK), block (32, RENDER_LINES_PER_BLOCK): x = env (coalesced, as everywhere), one
// line per thread.  Small blocks on purpose: they have to find room on SMs that another env group's emulation kernel
// occupies.  The pending range stays in R_MISC; the env's next emulation launch starts from an empty one (machine_load),
// and an env that is skipped meanwhile (gbenv_step_masked) is skipped here as well.
#define RENDER_LINES_PER_BLOCK 4
__global__ void __launch_bounds__(32 * RENDER_LINES_PER_BLOCK) k_render_pending(DevArrays d, const uint8_t *skip) {
    // the line buffer and the sprite sort keys are thread-local (L1-resident local memory), NOT shared memory: a kernel that
    // wants a different shared-memory carve-out cannot share an SM with the other group's emulation kernel
    uint32_t line[FB_LINE_WORDS], keys[10];
    const int tile = blockIdx.x, lane = threadIdx.x, env = tile * GB_TILE + lane;
    if (env >= d.n_envs || (skip && skip[env])) return;
    render_pending_lines(d, tile, lane, blockIdx.y * RENDER_LINES_PER_BLOCK + threadIdx.y, 144, line, keys, 1);
}
#endif

// ---------------------------------------------------------------------------------------------
// grid: (ceil(n / 32), ceil(IMG_WORDS / 8)); block (32, 8): x = env slot (coalesced), y = image word
__global__ void k_scatter_image(DevArrays d, const uint32_t *image, const int32_t *env_ids, int n, int version) {
    int i = blockIdx.x * 32 + threadIdx.x;
    uint32_t j = blockIdx.y * 8 + threadIdx.y;
    if (i >= n || j >= IMG_WORDS) return;
    int env = env_ids ? env_ids[i] : i;
    uint32_t v = image[j];
    uint32_t *slot = image_slot(d, env, j);
    if (j >= IMG_REGS) v = merge_loaded_reg(j - IMG_REGS, *slot, v, version, image[IMG_REGS + R_LCD0] & 0xFF);
    *slot = v;
}

__global__ void k_gather_image(DevArrays d, uint32_t *image, int env) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < IMG_WORDS) image[j] = *image_slot(d, env, j);
}

// PyBoy.get_memory_value / set_memory_value for one env: full bus semantics incl. IO side effects
__global__ void k_bus_access(DevArrays d, int env, uint32_t addr, uint32_t n, uint8_t *buf, int write) {
    if (threadIdx.x || blockIdx.x) return;
    Machine m;
    machine_load(m, d, env >> 5, env & 31);
    for (uint32_t i = 0; i < n; i++) {
        if (write) bus_write(m, (addr + i) & 0xFFFF, buf[i]);
        else buf[i] = (uint8_t)bus_read(m, (addr + i) & 0xFFFF);
    }
    if (write) machine_store(m, d, env >> 5, env & 31);
}

// PyBoy.send_input applied to every env at once (Interaction.key_event + IF bit 4 on a 1->0 edge)
__global__ void k_send_input(DevArrays d, int button, int pressed) {
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= d.n_envs) return;
    int tile = env >> 5, lane = env & 31;
    uint32_t *rj = d.regs + il_index(tile, R_WORDS, R_JOY, lane), *ri = d.regs + il_index(tile, R_WORDS, R_INT, lane);
    uint32_t w = *rj, dir = w & 0xFF, std_ = (w >> 8) & 0xFF;
    uint32_t bit = 1u << (button & 3);
    uint32_t &reg = button < 4 ? dir : std_;
    uint32_t before = reg;
    reg = pressed ? (reg & ~bit) : (reg | bit);
    if ((before ^ reg) & before) *ri |= IRQ_JOYPAD << 16;
    *rj = (w & 0xFFFF0000u) | dir | (std_ << 8);
}

// Test hook: Renderer.scanline + scanline_sprites for all 144 lines of one env, driven by the stored
// per-scanline parameters (PPU known-answer vectors: a save-state embeds the frame PyBoy rendered from
// exactly these inputs).
__global__ void k_debug_render_frame(DevArrays d, int env) {
    __shared__ uint32_t s_line[FB_LINE_WORDS], s_keys[10];
    if (threadIdx.x || blockIdx.x) return;
    Machine m;
    machine_load(m, d, env >> 5, env & 31);
    const uint32_t scroll = m.scroll, lcdc = m.lcdc;
    m.ly_window = -1;
    for (uint32_t y = 0; y < 144; y++) {
        uint2 v = m.lp[y << 5];
        m.scroll = v.x;
        m.lcdc = (lcdc & ~0x10u) | (v.y & 0x10);
        render_line(m, y, s_line, s_keys, 1);
    }
    m.scroll = scroll; m.lcdc = lcdc;
    machine_store(m, d, env >> 5, env & 31);
}
