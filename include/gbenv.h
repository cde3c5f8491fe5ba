/*
 * gbenv.h -- C ABI of the B200-native batched Game Boy environment (libgbenv.so).
 *
 * The reference has no FFI layer: its boundary is the Python class `pokegym.Environment`
 * (/root/reference/pokegym/__init__.py:1, environment.py:436-1812) sitting on PyBoy's Python API
 * (/root/reference/pokegym/pyboy_binding.py:42-91).  Each entry point below names the reference
 * interface it replaces; INTEGRATION.md shows the ctypes binding a pokegym maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative GBENV_E_* code on failure; nothing throws
 *     across the ABI; gbenv_last_error() returns a static/handle-owned message.
 *   - "dev" pointers are CUDA device pointers owned by the caller (e.g. PyTorch tensors);
 *     "host" pointers are ordinary host memory.  The library owns all emulator state.
 *   - a handle is bound to one CUDA device.  Entry points with a `stream` argument (a cudaStream_t passed
 *     as void*; NULL = the legacy default stream, which is what PyTorch uses by default) queue their
 *     work on that stream; the others use the handle's own stream.  Whatever the streams, calls on one
 *     handle take effect in CALL ORDER: when consecutive calls use different streams the later stream
 *     waits for an event recorded on the earlier one.  Calls are asynchronous with respect to the host
 *     unless stated otherwise.  Not re-entrant per handle.
 *   - there is NO CPU fallback: gbenv_create fails with GBENV_E_CUDA when no device is usable.
 *
 * The test oracle (oracle/liboracle.so) exports the same symbols with the prefix `oracle_`
 * operating on host memory, so one test body drives both.
 */
#ifndef GBENV_H
#define GBENV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GBENV_ABI_VERSION 7 /* 2: info row widened from 64 to 72 doubles; 3: gbenv_reset_dev, gbenv_submit_host / gbenv_fetch_host, gbenv_check, gbenv_step_masked;
                               4: gbenv_counts_map_sum, gbenv_reduce_info_masked; 5: gbenv_capture_frames, gbenv_frames_to_rgb;
                               6: gbenv_event_flags; 7: gbenv_step_packed, gbenv_reset_packed, gbenv_unpack_obs */

#define GBENV_STATE_BYTES 142610 /* PyBoy v9 save-state length (SURVEY.md 8c)              */
#define GBENV_OBS_H 72           /* environment.py:154-166: (144//2, 160//2, 4) uint8       */
#define GBENV_OBS_W 80
#define GBENV_OBS_C 4
#define GBENV_OBS_BYTES (GBENV_OBS_H * GBENV_OBS_W * GBENV_OBS_C)
#define GBENV_SCREEN_H 144
#define GBENV_SCREEN_W 160
#define GBENV_FRAME_WORDS 1440 /* packed frame: 144 lines x 10 words of 16 2-bit pixels (gbenv_capture_frames) */
#define GBENV_OBS_PACKED_WORDS 576  /* packed observation: 72 rows x 8 uint32 words (gbenv_step_packed)          */
#define GBENV_OBS_PACKED_BYTES 2304
#define GBENV_NUM_ACTIONS 8 /* pyboy_binding.ACTIONS :40  Down Left Right Up A B Start Select */
#define GBENV_ACT_FREQ 24   /* pyboy_binding.run_action_on_emulator :72 frame_skip=24         */
#define GBENV_INFO_SCALARS 72
#define GBENV_EVENT_FLAGS 130 /* entries of the reference's event table (gbenv_event_flags)                       */
#define GBENV_EVENT_WORDS 5   /* uint32 words of one env's event flags: GBENV_EVENT_FLAGS bits rounded up to 32 */

enum {
    GBENV_OK = 0,
    GBENV_E_ARG = -1,    /* bad argument (null handle, env out of range, bad length ...)     */
    GBENV_E_STATE = -2,  /* unsupported / malformed save-state blob                          */
    GBENV_E_CUDA = -3,   /* CUDA runtime error (message in gbenv_last_error)                 */
    GBENV_E_NOMEM = -4,  /* allocation failed                                                */
    GBENV_E_FAULT = -5   /* an env executed an illegal opcode (PyBoy would have raised)      */
};

typedef struct gbenv gbenv_t;

/* ---- lifetime ------------------------------------------------------------------------------
 * replaces pyboy_binding.make_env (:42-57) + Environment.__init__ (environment.py:102-197,437-511)
 * for n_envs instances at once.  `rom` is copied to the device (shared by all envs).            */
int gbenv_create(int n_envs, const uint8_t *rom_host, size_t rom_len, int device_id, gbenv_t **out);
int gbenv_destroy(gbenv_t *h); /* Environment.close (:412-413) */
const char *gbenv_last_error(const gbenv_t *h);
int gbenv_num_envs(const gbenv_t *h);
int gbenv_abi_version(void);
int gbenv_sync(gbenv_t *h); /* cudaStreamSynchronize on the handle's stream */
/* gbenv_sync + the sticky error state of the exploration storage.  Visited bitmaps (seen_coords / screen_memory,
 * environment.py:256-274, :1344) and heat maps (counts_map, :648-679) are paged out of pools shared by all envs, so any
 * env may hold all 248 maps; should a pool run dry the affected env stops matching the reference, which is an ERROR:
 * this call, and every gbenv_step / gbenv_reset* issued once the condition has reached the host (at most two calls
 * later, no synchronisation involved), return GBENV_E_NOMEM with the pool named in gbenv_last_error.             */
int gbenv_check(gbenv_t *h);
/* Tuning knob: envs carried by each warp of the emulation kernel (1..32).  The default is
 * chosen from n_envs and the SM count so that a small batch still fills the GPU with warps.        */
int gbenv_set_lanes_per_warp(gbenv_t *h, int lanes);
int gbenv_get_lanes_per_warp(const gbenv_t *h); /* the value in use (>= 1), or a negative error code */

/* ---- (4) reset from PyBoy .state files ------------------------------------------------------
 * replaces pyboy_binding.open_state_file / load_pyboy_state (:59-69).  A blob is parsed ONCE on
 * the host into a device-resident template; loading broadcasts the template into env state.     */
int gbenv_add_state_template(gbenv_t *h, const uint8_t *blob_host, size_t len, int *template_id_out);
/* PyBoy.load_state for the listed envs (env_ids_host == NULL: all envs). */
int gbenv_load_template(gbenv_t *h, const int32_t *env_ids_host, int n, int template_id);
/* Environment.__init__ `initial_states = [open_state_file(state_path)]` (environment.py:122):
 * the template gbenv_reset loads on an env's FIRST reset only (environment.py:1241-1242).       */
int gbenv_set_initial_template(gbenv_t *h, const int32_t *env_ids_host, int n, int template_id);
/* Fresh post-boot DMG machine (our convention for ROM-only runs; PyBoy would run its boot ROM). */
int gbenv_power_on(gbenv_t *h, const int32_t *env_ids_host, int n);
/* PyBoy.save_state: v9 blob of one env, synchronous. */
int gbenv_save_state(gbenv_t *h, int env, uint8_t *blob_host /* GBENV_STATE_BYTES */);

/* ---- (1)+(2) emulator: tick loop + PPU ------------------------------------------------------
 * replaces pyboy_binding.run_action_on_emulator (:71-91): press, 24 x tick (release before tick 8,
 * rendering enabled for the last tick only).  actions_dev: uint8[n_envs] in 0..7.               */
int gbenv_run_action(gbenv_t *h, const uint8_t *actions_dev, int frame_skip, void *stream);
/* PyBoy.tick() x n_frames without input; render: 0 = renderer disabled, 1 = enabled all frames. */
int gbenv_tick(gbenv_t *h, int n_frames, int render, void *stream);
/* PyBoy.send_input for every env: button 0..7 = Right Left Up Down A B Select Start.            */
int gbenv_send_input(gbenv_t *h, int button, int pressed, void *stream);
/* PyBoy.get_memory_value / set_memory_value (bus semantics incl. IO side effects), synchronous. */
int gbenv_read_mem(gbenv_t *h, int env, uint32_t addr, uint32_t n, uint8_t *out_host);
int gbenv_write_mem(gbenv_t *h, int env, uint32_t addr, uint32_t n, const uint8_t *in_host);
/* botsupport screen().screen_ndarray(): uint8[144*160*3] of one env, synchronous.               */
int gbenv_screen(gbenv_t *h, int env, uint8_t *rgb_host);
/* Batched, asynchronous frames (the reference's save_video / render() frames, pyboy_binding.py:77-78,86-87).
 * A PACKED frame is the env's framebuffer as the library stores it: 144 lines x 10 uint32 words = GBENV_FRAME_WORDS words
 * (5,760 B, 12x smaller than RGB, lossless).  The pixel (x, y) is the 2-bit shade at bit 2*(x & 15) of word y*10 + x/16;
 * the grey of shade s is {0xFF, 0x99, 0x55, 0x00}[s].
 * gbenv_capture_frames: the current frame of the listed envs into frames_dev uint32[n][GBENV_FRAME_WORDS].  env_ids_dev:
 * int32[n] on the device, any order, duplicates allowed; NULL means envs 0..n-1 (n <= n_envs).  A row whose id is outside
 * [0, n_envs) is left untouched and nothing is read for it.  For a valid id the row is bit-identical to the framebuffer
 * gbenv_screen decodes.  Asynchronous on `stream` and ordered after earlier calls on the handle.
 * gbenv_frames_to_rgb: n_frames packed frames -> out_dev uint8[n_frames][144][160][channels], channels 1 = grey, 3 = RGB as
 * gbenv_screen.  out_dev must be 16-byte aligned.  Asynchronous on `stream`.
 * Both: GBENV_E_ARG on NULL or misaligned buffers, a negative count, channels not 1 or 3, NULL ids with n > n_envs; a count
 * of 0 is a successful no-op.                                                                   */
int gbenv_capture_frames(gbenv_t *h, const int32_t *env_ids_dev, int n, uint32_t *frames_dev, void *stream);
int gbenv_frames_to_rgb(gbenv_t *h, const uint32_t *frames_dev, int n_frames, int channels, uint8_t *out_dev, void *stream);

/* ---- (3) Environment.reset / step with fused reward + observation ---------------------------
 * gbenv_reset == Environment.reset (environment.py:1233-1334) for envs with mask[e] != 0
 * (mask_host == NULL: all).  obs_dev: uint8[n_envs][obs_stride] (obs_stride >= GBENV_OBS_BYTES),
 * only rows of reset envs are written.
 * Guarantee of every gbenv_reset* call: an env's info row (gbenv_get_info) is left as its last step wrote it, and its heat
 * map keeps accumulating (it lives as long as the env).  So after an auto-reset on the `done` of a step, the info rows of
 * the envs that just finished are still there for gbenv_reduce_info_masked(mask = that done).  The CPU oracle differs
 * here: its reset zeroes the row (DESIGN.md section 2).                                         */
int gbenv_reset(gbenv_t *h, const uint8_t *mask_host, int max_episode_steps, double reward_scale,
                uint8_t *obs_dev, size_t obs_stride, void *stream);
/* The same with a DEVICE mask (e.g. the `done` vector gbenv_step just wrote): nothing touches the host, so a vectoriser
 * can auto-reset finished envs without a round trip.  Which envs still have their first reset -- the one that loads
 * their save-state, environment.py:1241-1242 -- ahead of them is tracked on the device.                       */
int gbenv_reset_dev(gbenv_t *h, const uint8_t *mask_dev, int max_episode_steps, double reward_scale,
                    uint8_t *obs_dev, size_t obs_stride, void *stream);
/* gbenv_step == Environment.step (environment.py:1336-1812) for every env:
 *   actions_dev uint8[n]; obs_dev uint8[n][obs_stride] (a slice of the rollout tensor);
 *   reward_dev double[n] (the reference returns Python floats); done_dev uint8[n]
 *   (terminated == truncated, environment.py:1613,1812).  No host round trip.                   */
int gbenv_step(gbenv_t *h, const uint8_t *actions_dev, uint8_t *obs_dev, size_t obs_stride,
               double *reward_dev, uint8_t *done_dev, void *stream);
/* The same for the envs with skip_dev[e] == 0 only (skip_dev NULL: all).  A skipped env is not emulated: its state, info row
 * and observation row stay untouched and it reports reward 0, done 0.  This is what a vectoriser needs that resets an env on
 * the call AFTER its `done` and ignores that call's action for it (PufferLib's Serial / Multiprocessing backends):
 * gbenv_reset_dev(mask = previous done) followed by gbenv_step_masked(skip = the same mask).                          */
int gbenv_step_masked(gbenv_t *h, const uint8_t *actions_dev, const uint8_t *skip_dev, uint8_t *obs_dev, size_t obs_stride,
                      double *reward_dev, uint8_t *done_dev, void *stream);
/* Packed observations: the reference observation stored losslessly in GBENV_OBS_PACKED_BYTES (2,304 B, 10x less than
 * GBENV_OBS_BYTES), for rollout buffers that would not fit in device memory otherwise.  Channels 0-2 of the reference
 * observation are the same grey, one of four levels, and channel 3 is 0 or 255, so a pixel is 3 bits.
 * Layout of one env's uint32[GBENV_OBS_PACKED_WORDS]: obs row i (0..71) is words 8i .. 8i+7.
 *   - words 8i+k, k = 0..4: obs pixels j = 16k .. 16k+15, the 2-bit shade of pixel j at bit 2*(j & 15) (the convention of the
 *     packed frame above).  The shade of obs pixel (i, j) is the framebuffer's at (x = 2j, y = 2i); channels 0-2 are
 *     {0xFF, 0x99, 0x55, 0x00}[shade].
 *   - words 8i+5+m, m = 0..2: the visited bit of pixel j = 32m + b at bit b; channel 3 is 255 when it is set, 0 otherwise.
 *     Bits of j >= 80 are 0.
 * gbenv_step_packed is gbenv_step_masked with the observation written to packed_dev uint32[n_envs][GBENV_OBS_PACKED_WORDS]:
 * skipped envs' rows are untouched, and rewards, dones, info rows and emulator state are those gbenv_step_masked gives.
 * gbenv_reset_packed is gbenv_reset_dev with packed output: only the rows of reset envs are written (mask_dev NULL: all).
 * gbenv_unpack_obs turns n packed rows into out_dev uint8[n][GBENV_OBS_BYTES], the bytes gbenv_step would have written.  It
 * reads no emulator state, so rows of any step or rollout slot can be decoded; asynchronous on `stream`.
 * All three: rows are contiguous; packed_dev / out_dev must be 16-byte aligned.  GBENV_E_ARG on a NULL or misaligned buffer
 * or n < 0; n == 0 is a successful no-op.  Streams and call order as for the calls above.  The host-buffer calls below keep
 * the reference format.                                                                          */
int gbenv_step_packed(gbenv_t *h, const uint8_t *actions_dev, const uint8_t *skip_dev, uint32_t *packed_dev, double *reward_dev,
                      uint8_t *done_dev, void *stream);
int gbenv_reset_packed(gbenv_t *h, const uint8_t *mask_dev, int max_episode_steps, double reward_scale, uint32_t *packed_dev, void *stream);
int gbenv_unpack_obs(gbenv_t *h, const uint32_t *packed_dev, int n, uint8_t *out_dev, void *stream);
/* Same call with HOST buffers (pinned or pageable): copies in, steps, copies out, synchronises.
 * This is the reference-facing entry point a pokegym worker would call.                         */
int gbenv_step_host(gbenv_t *h, const uint8_t *actions_host, uint8_t *obs_host, double *reward_host,
                    uint8_t *done_host);
int gbenv_reset_host(gbenv_t *h, const uint8_t *mask_host, int max_episode_steps, double reward_scale,
                     uint8_t *obs_host);
/* Two-call form of gbenv_step_host: submit queues the step and returns at once, fetch blocks until the results of the
 * OLDEST queued step are in the host buffers given to its submit.  Up to two steps may be in flight, so that the
 * device-to-host copy of step t (23 KB per env) overlaps the emulation of step t+1.  Buffers should be pinned.   */
int gbenv_submit_host(gbenv_t *h, const uint8_t *actions_host, uint8_t *obs_host, double *reward_host,
                      uint8_t *done_host);
int gbenv_fetch_host(gbenv_t *h);
/* Episode-info scalars (environment.py:1621-1810 `stats` / `reward` numeric entries), one row of
 * GBENV_INFO_SCALARS doubles per env, written to info_dev[n][GBENV_INFO_SCALARS].               */
int gbenv_get_info(gbenv_t *h, double *info_dev, void *stream);
/* Sum of the info rows over envs (+ env count in slot 0): the vector ranks all-reduce over NCCL. */
int gbenv_reduce_info(gbenv_t *h, double *sum_dev /* GBENV_INFO_SCALARS */, void *stream);
/* gbenv_reduce_info over the envs with mask_dev[e] != 0 only (mask_dev NULL: all envs, bit-identical to gbenv_reduce_info);
 * slot 0 = number of those envs that have stepped at least once.  The mean a trainer logs when episodes end is this sum
 * with mask = the `done` of the step, divided by slot 0.  Asynchronous on `stream`.                                 */
int gbenv_reduce_info_masked(gbenv_t *h, const uint8_t *mask_dev, double *sum_dev /* GBENV_INFO_SCALARS */, void *stream);
/* `pokemon_exploration_map` (environment.py:448,648-679,1624): int32[444*436] of one env, synchronous.  Heat maps are
 * paged (DESIGN.md section 3): per env a directory of 28 x 28 blocks of 16 x 16 cells, blocks taken from a pool shared by
 * all envs on first touch; this call rebuilds the dense image.  GBENV_COUNTS_MAP=0 switches heat maps off (this call then
 * fails with GBENV_E_ARG); GBENV_COUNTS_BLOCKS sizes the pool, and a pool that runs dry is reported by gbenv_check.  */
int gbenv_counts_map(gbenv_t *h, int env, int32_t *map_host);
/* Sum of the heat maps of the envs with mask_dev[e] != 0 (mask_dev NULL: all envs) into sum_dev int64[444*436], which is
 * overwritten: each cell is the plain integer sum of that cell over those envs' maps, -1 marks included (the reference
 * trainer's exploration overlay sums the `pokemon_exploration_map`s of the envs that finished, environment.py:1624).
 * Asynchronous on `stream`, ordered after earlier calls on the handle.  GBENV_E_ARG when heat maps are switched off;
 * GBENV_E_NOMEM once an exhausted pool has been reported (as gbenv_step), since the maps are then incomplete.        */
int gbenv_counts_map_sum(gbenv_t *h, const uint8_t *mask_dev, int64_t *sum_dev /* 444*436 */, void *stream);
/* The event flags behind the `*_events_aggregate` / `gym_events` and `detailed_rewards_*` entries of the info dict
 * (environment.py:1621-1810, ram_map_leanke.py monitor_*_events) for a list of envs, into flags_dev uint32[n][GBENV_EVENT_WORDS].
 * Bit k & 31 of word k >> 5 is the WRAM bit that entry k of the reference's event table reads, as stored, whatever the sign
 * of its weight.  The table has GBENV_EVENT_FLAGS entries in the order of pokegym_b200/event_table.json: silph_co 53,
 * dojo 8, hideout 15, poke_tower 17, gym3 .. gym7.  Entries that read the same bit (gym 5's and gym 6's leader, D7B3 bit 1)
 * each keep their own position; bits 130..159 are 0.  This is that table and nothing else: there is no address or length,
 * and it is not a RAM read (gbenv_read_mem reads one env's bytes).
 * env_ids_dev: int32[n] on the device, any order, duplicates allowed; NULL means envs 0..n-1 (n <= n_envs).  A row whose id
 * is outside [0, n_envs) is left untouched and nothing is read for it.  Asynchronous on `stream`, ordered after earlier
 * calls on the handle.  GBENV_E_ARG on a NULL handle, a NULL or misaligned output with n > 0, n < 0, or NULL ids with
 * n > n_envs; n == 0 is a successful no-op.                                                                            */
int gbenv_event_flags(gbenv_t *h, const int32_t *env_ids_dev, int n, uint32_t *flags_dev, void *stream);

/* ---- diagnostics ----------------------------------------------------------------------------*/
typedef struct gbenv_counters {
    uint64_t instructions; /* SM83 instructions executed, all envs, since create */
    uint64_t cycles;       /* emulated T-cycles, all envs                        */
    uint64_t frames;       /* emulated frames, all envs                          */
    uint64_t faults;       /* envs that hit an illegal opcode                    */
    uint64_t kernel_launches;
} gbenv_counters_t;
int gbenv_get_counters(gbenv_t *h, gbenv_counters_t *out);
/* Device time of the kernels launched by the last gbenv_step/gbenv_run_action call, measured with
 * CUDA events on the launching stream (ms).  which: 0 = emulate, 1 = obs/reward.  Synchronous.  */
int gbenv_last_kernel_ms(gbenv_t *h, int which, float *ms_out);
/* Running total of the same device times over every gbenv_step since create (CUDA events recorded on
 * the launching stream around each kernel group; folding is lazy, so the step path never blocks).    */
int gbenv_kernel_time_total(gbenv_t *h, int which, double *ms_total_out, uint64_t *steps_out);
/* Non-serialised core fields (STATRegister._mode, Renderer.ly_window ...) for parity checks.    */
typedef struct gbenv_core_extra {
    int32_t stat_mode;
    int32_t ly_window;
    int32_t fault;
    int32_t reserved;
} gbenv_core_extra_t;
int gbenv_get_core_extra(gbenv_t *h, int env, gbenv_core_extra_t *out);
/* Test hook for the PPU known-answer vectors: re-render all 144 lines of one env from its current VRAM /
 * OAM / palettes using the stored per-scanline parameters (what PyBoy's renderer did for the frame a
 * save-state embeds), into the env's framebuffer.  Synchronous.                                      */
int gbenv_debug_render_frame(gbenv_t *h, int env);

#ifdef __cplusplus
}
#endif
#endif /* GBENV_H */
