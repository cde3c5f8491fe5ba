// gb_wrap.cuh -- fused reward extraction, RAM side effects and observation assembly on the device.
//
// Replaces the Python half of pokegym's hot path, evaluated over device RAM with no host readback:
//   /root/reference/pokegym/environment.py  reset :1233-1334, step :1338-1613, render :256-274
//   /root/reference/pokegym/ram_map.py :1522-1601,1858-1898   ram_map_leanke.py :793-1098
//   /root/reference/pokegym/game_map.py :11-18                red_ram_api.py :59-73 (RAM side effects)
// Reward arithmetic is float64 in the reference's own association order, so results are bit-identical.
//
// k_wrap_step   : one thread per env (lane == env inside a tile, so the 32 envs of a warp read the same
//                 WRAM addresses as whole 128-byte lines): reward, done, RAM writes, visited bitmap.
// k_wrap_obs    : one block per 32-env tile: transposes the 2-bpp framebuffer through shared memory and
//                 writes uint8[72,80,4] rows straight into the caller's rollout tensor, 320 contiguous
//                 bytes per env row, with channel 3 cut from the visited bitmap.
#pragma once
#include "../../include/gbenv.h"
#include "../../include/gbenv_info.h"
#include "gb_device.cuh"

#define WRAP_CUT_COORDS 64
#define COUNTS_H 444
#define COUNTS_W 436
#define CM_BLOCK 16                           // heat-map blocks of 16 x 16 cells = 1 KiB
#define CM_BLOCKS_X ((COUNTS_W + CM_BLOCK - 1) / CM_BLOCK)
#define CM_BLOCKS_Y ((COUNTS_H + CM_BLOCK - 1) / CM_BLOCK)
#define CM_DIR_ENTRIES (CM_BLOCKS_X * CM_BLOCKS_Y)
// WrapArrays.ctl words
#define CTL_VIS_FREE 0    // number of free visited-bitmap pages (top of the free stack)
#define CTL_CM_NEXT 1     // next never-used heat-map block
#define CTL_ERROR 2       // sticky error bits, see GBENV_POOL_*
#define POOL_ERR_VISITED 1u
#define POOL_ERR_HEATMAP 2u
#define POOL_ERR_CUT_COORDS 4u

struct CutCoord {
    int32_t x, y, map, pad;
    double value;
};

// per-env wrapper state (AoS: touched by one thread per step)
struct WrapState {
    // env-lifetime
    int32_t reset_count, is_dead, last_map, initial_template;
    double item_reward[5];
    long long coord_sum;  // running np.sum(counts_map)
    // per-episode
    int32_t time, max_episode_steps, have_last_reward, overflow;
    double reward_scale, last_reward, last_delta, total_healing, last_hp;
    int32_t max_events, max_level_sum, max_opponent_level, n_seen_coords;
    int32_t n_seen_maps, prev_map_n, death_count, last_party_size;
    int32_t hm_latch, cut, used_cut, n_cut_coords;
    int32_t n_cut_tiles, n_cut_state, seen_start_menu, seen_pokemon_menu;
    int32_t seen_stats_menu, seen_bag_menu, last_map_id_plus1, pad0;
    int32_t reset_r, reset_c, reset_map, reset_pending;  // render() at reset marks a tile seen_coords does not hold
    int32_t cut_state[3][6];
    uint32_t seen_maps_bits[8], cut_tiles_bits[8], moves_bits[6];
    CutCoord cut_coords[WRAP_CUT_COORDS];
};

// Exploration storage is paged: nothing is reserved per env, so ANY env can hold all 248 maps / the whole 444 x 436 heat map
// as long as the shared pools last (they are sized to the batch or to a memory budget, gbenv.cu); a pool running dry is an
// error (CTL_ERROR, reported by the next gbenv_step / gbenv_reset / gbenv_check), never a silent loss.
//   visited bitmaps (seen_coords / screen_memory, environment.py:256-274, :1344): per env a page table of 248 maps x 4 row bands;
//     pages come from a free stack and go back to it, zeroed, when the env is reset.
//   heat map (counts_map, :648-679, env-lifetime): per env a directory of 28 x 28 blocks; blocks are bump-allocated, never freed.
struct WrapArrays {
    WrapState *state;     // [n_envs]
    uint32_t *vis_pt;     // [n_envs][VIS_PT_ENTRIES]: page index + 1, 0 = no page yet
    uint32_t *vis_pool;   // [vis_pages][VIS_PAGE_WORDS]
    int32_t *vis_free;    // [vis_pages] stack of free page indices
    uint32_t *cm_dir;     // [n_envs][CM_DIR_ENTRIES]: block index + 1, 0 = no block yet; null = heat maps switched off
    int32_t *cm_pool;     // [cm_blocks][CM_BLOCK * CM_BLOCK]
    int32_t *ctl;         // CTL_* words
    int vis_pages, cm_blocks;
};

struct MapOffset { int16_t x, y, known; };
__constant__ MapOffset c_map_offsets[WRAP_MAPS] = {
#include "map_offsets.inc"
};

// environment.py:58-78 TREE_POSITIONS_PIXELS (first, second, map)
__constant__ int c_trees[19][3] = {
    {3184, 3584, 6},  {3375, 3391, 6},  {2528, 3616, 134}, {2480, 3568, 134}, {2560, 3584, 134}, {1104, 2944, 13}, {1264, 3136, 13},
    {1216, 3616, 13}, {1216, 3744, 13}, {1216, 3872, 13},  {1088, 4000, 1},   {992, 4288, 1},    {3984, 4512, 5},  {4640, 1392, 36},
    {4464, 2176, 20}, {5488, 2336, 21}, {5488, 2368, 21},  {5488, 2400, 21},  {5488, 2432, 21}};

// red_memory_menus.py:237-299: keys of TEXT_MENU_CURSOR_LOCATIONS as CC30 | CC31 << 8
__constant__ uint16_t c_cursor_keys[48] = {
    0xC3D3, 0xC3FB, 0xC423, 0xC44B, 0xC473, 0xC49B, 0xC4C3, 0xC44C, 0xC474, 0xC3B5, 0xC3DD, 0xC405, 0xC3C9, 0xC3F1, 0xC419, 0xC441,
    0xC49A, 0xC4C2, 0xC4EA, 0xC4C1, 0xC4A9, 0xC4BD, 0xC4D1, 0xC4E5, 0xC4C7, 0xC3B4, 0xC3DC, 0xC404, 0xC42C, 0xC454, 0xC47C, 0xC49C,
    0xC4C4, 0xC4EC, 0xC4E9, 0xC48A, 0xC4B2, 0xC3F5, 0xC41D, 0xC445, 0x0169, 0xC4EF, 0xC44F, 0xC477, 0xC469, 0xC459, 0xC46D, 0xC481};

// ram_map_leanke.py monitor_* dicts in insertion order (event_bits.inc): address | bit << 16 | (weight & 0xFF) << 24
#define EV(a, b, w) ((uint32_t)(a) | ((uint32_t)(b) << 16) | ((uint32_t)((w) & 0xFF) << 24))
__constant__ uint32_t c_events[] = {
#include "event_bits.inc"
};
#undef EV
// group boundaries inside c_events: silph, dojo, hideout, tower, gym3..7
__constant__ int c_event_groups[10] = {0, 53, 61, 76, 93, 99, 107, 114, 122, 130};

__device__ __forceinline__ uint32_t RAM(Machine &m, uint32_t a) { return bus_read(m, a); }
__device__ __forceinline__ uint32_t RBIT(Machine &m, uint32_t a, uint32_t b) { return (bus_read(m, a) >> b) & 1; }

// environment.py:1201-1219 calculate_event_rewards(base 10, increment 2, multiplier 1)
__device__ inline int event_group_reward(Machine &m, int g) {
    int total = 0, cur = 10;
    for (int i = c_event_groups[g]; i < c_event_groups[g + 1]; i++) {
        uint32_t e = c_events[i];
        int points = (int)(int8_t)(e >> 24) * (int)RBIT(m, e & 0xFFFF, (e >> 16) & 7);
        if (points > 0) {
            total += cur * points;
            cur += 2;
        }
    }
    return total;
}

__device__ __forceinline__ void wrap_position(Machine &m, int &r, int &c, int &map_n) {  // ram_map.position :1522-1538
    r = (int)RAM(m, 0xD361);
    c = (int)RAM(m, 0xD362);
    map_n = (int)RAM(m, 0xD35E);
    if (map_n > 247) map_n = 247;
}

// visited bitmap: the 8 words of row r of map map_n, its page allocated on first use (nullptr: no page / pool exhausted)
__device__ inline uint32_t *visited_row(const WrapArrays &w, WrapState &s, int env, int map_n, int r, bool create) {
    uint32_t *e = w.vis_pt + (size_t)env * VIS_PT_ENTRIES + map_n * VIS_BANDS + (r / VIS_BAND_ROWS);
    uint32_t pg = *e;
    if (!pg) {
        if (!create) return nullptr;
        const int i = atomicSub(&w.ctl[CTL_VIS_FREE], 1);  // pops only in this kernel family; pushes only in k_vis_release
        if (i <= 0) {
            atomicAdd(&w.ctl[CTL_VIS_FREE], 1);
            atomicOr((unsigned int *)&w.ctl[CTL_ERROR], POOL_ERR_VISITED);
            s.overflow = 1;
            return nullptr;
        }
        pg = (uint32_t)w.vis_free[i - 1] + 1;
        *e = pg;
    }
    return w.vis_pool + (size_t)(pg - 1) * VIS_PAGE_WORDS + (r % VIS_BAND_ROWS) * VIS_ROW_WORDS;
}

// heat map cell (glob_r, glob_c) of env, its block allocated on first use
__device__ inline int32_t *heat_cell(const WrapArrays &w, WrapState &s, int env, int glob_r, int glob_c) {
    uint32_t *e = w.cm_dir + (size_t)env * CM_DIR_ENTRIES + (glob_r / CM_BLOCK) * CM_BLOCKS_X + (glob_c / CM_BLOCK);
    uint32_t b = *e;
    if (!b) {
        const int i = atomicAdd(&w.ctl[CTL_CM_NEXT], 1);
        if (i >= w.cm_blocks) {
            atomicSub(&w.ctl[CTL_CM_NEXT], 1);
            atomicOr((unsigned int *)&w.ctl[CTL_ERROR], POOL_ERR_HEATMAP);
            s.overflow = 1;
            return nullptr;
        }
        b = (uint32_t)i + 1;
        *e = b;
    }
    return w.cm_pool + (size_t)(b - 1) * (CM_BLOCK * CM_BLOCK) + (glob_r % CM_BLOCK) * CM_BLOCK + (glob_c % CM_BLOCK);
}

__device__ __forceinline__ void victory_road_patch(Machine &m) {  // environment.py:1014-1025
    bus_write(m, 0xD7EE, RAM(m, 0xD7EE) | 0x81);
    bus_write(m, 0xD813, RAM(m, 0xD813) | 0x41);
    bus_write(m, 0xD869, RAM(m, 0xD869) | 0x80);
}

__device__ __forceinline__ void update_last_map_id(Machine &m, WrapState &s) {  // environment.py:1027-1052
    int cur = (int)RAM(m, 0xD35E) + 1;
    if (cur == s.last_map_id_plus1) return;
    s.last_map_id_plus1 = cur;
    int id = cur - 1;
    if (id == 0x6C || id == 0xC2 || id == 0xC6 || id == 0x22) victory_road_patch(m);
}

// render(): mark the current tile in screen_memory (environment.py:258-262)
__device__ inline void wrap_mark_render(const WrapArrays &w, WrapState &s, Machine &m, int env, bool at_reset) {
    int r, c, map_n;
    wrap_position(m, r, c, map_n);
    if (r > 254 || c > 254) return;
    uint32_t *row = visited_row(w, s, env, map_n, r, true);
    if (!row) return;
    uint32_t bit = 1u << (c & 31), *word = row + (c >> 5);
    if (at_reset) {
        s.reset_pending = !(*word & bit);
        s.reset_r = r; s.reset_c = c; s.reset_map = map_n;
    }
    *word |= bit;
}

// red_ram_api.py:59-73 Game.process_game_states: its only observable effect is the RAM clear at :596-600
__device__ inline void wrap_process_game_states(Machine &m) {
    if (RAM(m, 0xCFC4) != 0) return;
    uint32_t battle_type = RAM(m, 0xD057), pre_battle = RAM(m, 0xD059);
    if (battle_type || pre_battle) {
        uint32_t cur = RAM(m, 0xCC30) | (RAM(m, 0xCC31) << 8);
        for (int i = 0; i < 48; i++)
            if (c_cursor_keys[i] == cur) return;
        if (cur == 0 || !battle_type) return;
        if ((RAM(m, 0xD125) == 0x01 && RAM(m, 0xD730) != 0x40) || RAM(m, 0xCC52) == 0x00) return;
    }
    if (RAM(m, 0xCD38) != 0) return;
    bus_write(m, 0xCC30, 0);
    bus_write(m, 0xCC31, 0);
    for (uint32_t i = 0; i < 10; i++) bus_write(m, 0xCF7C + i, 0);
}

struct StepScalars {  // values of the current step needed by the info row
    int r, c, map_n, party_size, level_sum, max_level, badges, bill_state, hm_count, events, money, n_seen, n_caught, n_moves;
    int dojo_reward, bill_capt_rew, cut_rew;
    double level_reward, exploration_reward, tree_distance_reward, cut_coords, cut_tiles, start_menu, pokemon_menu, stats_menu, bag_menu;
    double reward, reward_abs;
};

// Everything Environment.step does after run_action_on_emulator (:1338-1613).  Returns the reward.
__device__ inline double wrap_after_emulation(const WrapArrays &w, WrapState &s, Machine &m, int env, int *done, StepScalars *out) {
    s.time += 1;
    int r, c, map_n;
    wrap_position(m, r, c, map_n);
    {  // seen_coords.add((r, c, map_n))  :1344-1345
        uint32_t *row = visited_row(w, s, env, map_n, r, true);
        if (row) {
            uint32_t bit = 1u << (c & 31), *word = row + (c >> 5);
            bool is_reset_tile = s.reset_pending && r == s.reset_r && c == s.reset_c && map_n == s.reset_map;
            if (!(*word & bit) || is_reset_tile) s.n_seen_coords++;
            if (is_reset_tile) s.reset_pending = 0;
            *word |= bit;
        }
    }
    wrap_process_game_states(m);  // :1348
    for (uint32_t i = 0; i < 20; i++) {  // :1349,1358-1372 (all 20 slots, no terminator check)
        uint32_t id = RAM(m, 0xD31E + 2 * i);
        if (id == 0x3E) s.item_reward[0] = 20.0;
        if (id == 0x48) s.item_reward[1] = 20.0;
        if (id == 0x4A) s.item_reward[2] = 20.0;
        if (id == 0x33) s.item_reward[3] = 20.0;
        if (id == 0x06) s.item_reward[4] = 20.0;
    }
    update_last_map_id(m, s);  // :1352
    double exploration_reward = (s.used_cut < 1 ? 0.02 : 0.1) * (double)s.n_seen_coords;  // :1375
    int glob_r = r + c_map_offsets[map_n].y, glob_c = c + c_map_offsets[map_n].x;          // game_map.py:11-18
    if (glob_r < COUNTS_H && glob_c < COUNTS_W) {  // update_heat_map :648-679
        const bool same_map = s.last_map == map_n || s.last_map == -1;
        int32_t *cell = w.cm_dir ? heat_cell(w, s, env, glob_r, glob_c) : nullptr;
        if (cell) {
            int32_t old = *cell, neu = same_map ? old + 1 : -1;
            *cell = neu;
            s.coord_sum += (long long)neu - old;
        }
    }
    s.last_map = map_n;
    if (map_n != s.prev_map_n) {  // :1378-1382
        s.prev_map_n = map_n;
        uint32_t bit = 1u << (map_n & 31);
        if (!(s.seen_maps_bits[map_n >> 5] & bit)) {
            s.seen_maps_bits[map_n >> 5] |= bit;
            s.n_seen_maps++;
        }
    }
    // :1386-1391 level reward
    int party_size = (int)RAM(m, 0xD163), level_sum = 0, max_level = 0;
    for (uint32_t k = 0; k < 6; k++) {
        int lv = (int)RAM(m, 0xD18C + 44 * k);
        level_sum += lv;
        max_level = lv > max_level ? lv : max_level;
    }
    if (level_sum > s.max_level_sum) s.max_level_sum = level_sum;
    double level_reward = s.max_level_sum < 50 ? (double)s.max_level_sum : 50.0 + (double)(s.max_level_sum - 50) / 4.0;
    // :1394-1408 healing / death
    int hp_sum = 0, max_hp_sum = 0;
    for (uint32_t k = 0; k < 6; k++) {
        hp_sum += 256 * (int)RAM(m, 0xD16C + 44 * k) + (int)RAM(m, 0xD16D + 44 * k);
        max_hp_sum += 256 * (int)RAM(m, 0xD18D + 44 * k) + (int)RAM(m, 0xD18E + 44 * k);
    }
    double hp = max_hp_sum == 0 ? 1.0 : (double)hp_sum / (double)max_hp_sum;
    double hp_delta = hp - s.last_hp;
    if (hp_delta > 0.2 && party_size == s.last_party_size && !s.is_dead) s.total_healing += hp_delta;
    if (hp <= 0 && s.last_hp > 0) {
        s.death_count += 1;
        s.is_dead = 1;
    } else if (hp > 0.01) {
        s.is_dead = 0;
    }
    s.last_hp = hp;
    s.last_party_size = party_size;
    // :1411-1426
    int badges = __popc(RAM(m, 0xD356));
    int bill_state = (int)RBIT(m, 0xD7F2, 3);
    uint32_t hm_mask = 0;
    for (uint32_t i = 0; i < 10; i++) {  // ram_map.get_items_in_bag :1867-1875
        uint32_t id = RAM(m, 0xD31E + 2 * i);
        if (id == 0 || id == 0xFF) break;
        if (id >= 0xC4 && id <= 0xC8) hm_mask |= 1u << (id - 0xC4);
    }
    int hm_count = __popc(hm_mask);
    if (hm_count >= 1 && s.hm_latch == 0) s.hm_latch = 1;
    int cut_rew = s.cut * 8;
    double tree_distance_reward = 0.0;  // detect_and_reward_trees :277-312 (player_x = glob_r, player_y = glob_c)
    for (int i = 0; i < 19; i++) {
        if (c_trees[i][2] != map_n) continue;
        int tree_x = c_trees[i][1] / 16, tree_y = c_trees[i][0] / 16;
        int cy = (tree_x == 212 && tree_y == 210) ? 211 : tree_y;
        int d = abs(glob_r - tree_x) + abs(glob_c - cy);
        if (d <= 5) tree_distance_reward += 1.0 / (double)(d > 1 ? d : 1);
    }
    int money;
    {
        uint32_t b0 = RAM(m, 0xD347), b1 = RAM(m, 0xD348), b2 = RAM(m, 0xD349);
        money = 10000 * (10 * (b0 >> 4) + (b0 & 15)) + 100 * (10 * (b1 >> 4) + (b1 & 15)) + (10 * (b2 >> 4) + (b2 & 15));
    }
    int max_opp = 0;
    for (uint32_t k = 0; k < 6; k++) {
        int lv = (int)RAM(m, 0xD8C5 + 44 * k);
        max_opp = lv > max_opp ? lv : max_opp;
    }
    if (max_opp > s.max_opponent_level) s.max_opponent_level = max_opp;
    // :1443-1445 events: popcount of D747..D885 minus 13 minus museum ticket, floor 0
    int num_events = 0;
    for (uint32_t a = 0xD747; a < 0xD886; a++) num_events += __popc(RAM(m, a));
    int events = num_events - 13 - (int)RBIT(m, 0xD754, 0);
    events = events < 0 ? 0 : events;
    if (events > s.max_events) s.max_events = events;
    int dojo_reward = 0;  // ram_map_leanke.dojo :793-814
    for (int i = c_event_groups[1]; i < c_event_groups[2]; i++) {
        uint32_t e = c_events[i];
        dojo_reward += (int)(int8_t)(e >> 24) * (int)RBIT(m, e & 0xFFFF, (e >> 16) & 7);
    }
    int silph_ev = event_group_reward(m, 0), dojo_ev = event_group_reward(m, 1), hideout_ev = event_group_reward(m, 2);
    int tower_ev = event_group_reward(m, 3), g3 = event_group_reward(m, 4), g4 = event_group_reward(m, 5);
    int g5 = event_group_reward(m, 6), g6 = event_group_reward(m, 7), g7 = event_group_reward(m, 8);
    // :1496-1538 cut state machine
    if (RAM(m, 0xD057) == 0 && s.cut == 1) {
        int dir = (int)RAM(m, 0xC109), x = (int)RAM(m, 0xD362), y = (int)RAM(m, 0xD361), map_id = (int)RAM(m, 0xD35E);
        int cx = x, cy = y;
        bool have_coords = true;
        if (dir == 0) cy = y + 1;
        else if (dir == 4) cy = y - 1;
        else if (dir == 8) cx = x - 1;
        else if (dir == 0xC) cx = x + 1;
        else have_coords = false;  // the reference raises UnboundLocalError if such a step ever matches
        if (s.n_cut_state == 3) {
            for (int k = 0; k < 6; k++) {
                s.cut_state[0][k] = s.cut_state[1][k];
                s.cut_state[1][k] = s.cut_state[2][k];
            }
            s.n_cut_state = 2;
        }
        int32_t *cs = s.cut_state[s.n_cut_state++];
        cs[0] = (int)RAM(m, 0xCFC6); cs[1] = (int)RAM(m, 0xCFCB); cs[2] = (int)RAM(m, 0xCD6A);
        cs[3] = (int)RAM(m, 0xD367); cs[4] = (int)RAM(m, 0xD125); cs[5] = (int)RAM(m, 0xCD3D);
        bool hit = false;
        double val = 0.0;
        if (s.n_cut_state == 3) {
            const int32_t(*q)[6] = s.cut_state;
            auto tail_is = [&](const int32_t *e, int a1, int a4) { return e[1] == a1 && e[2] == 1 && e[3] == 0 && e[4] == a4 && e[5] == 1; };
            // CUT_SEQ (:50): ((t,1,1,0,4,1),(t,1,1,0,1,1)) for t in {0x3D, 0x50} over the last two entries
            if ((q[1][0] == 0x3D || q[1][0] == 0x50) && q[2][0] == q[1][0] && tail_is(q[1], 1, 4) && tail_is(q[2], 1, 1)) {
                hit = true;
                val = 10.0;
            } else if (q[0][0] == 0x52 && q[1][0] == 0x52 && q[2][0] == 0x52 && tail_is(q[0], 255, 1) && tail_is(q[1], 255, 1) && tail_is(q[2], 1, 1)) {
                hit = true;  // CUT_GRASS_SEQ (:48)
                val = 0.001;
            } else {  // CUT_FAIL_SEQ (:49) with the tile id masked out
                auto fail_is = [&](const int32_t *e, int a4) { return e[1] == 255 && e[2] == 0 && e[3] == 0 && e[4] == a4 && e[5] == 1; };
                if (fail_is(q[0], 4) && fail_is(q[1], 1) && fail_is(q[2], 1)) {
                    hit = true;
                    val = 0.001;
                }
            }
        }
        if (hit && have_coords) {
            int i = 0;
            for (; i < s.n_cut_coords; i++)
                if (s.cut_coords[i].x == cx && s.cut_coords[i].y == cy && s.cut_coords[i].map == map_id) break;
            if (i < s.n_cut_coords) {
                s.cut_coords[i].value = val;
            } else if (s.n_cut_coords < WRAP_CUT_COORDS) {
                CutCoord &e = s.cut_coords[s.n_cut_coords++];
                e.x = cx; e.y = cy; e.map = map_id; e.value = val;
            } else {
                s.overflow = 1;
                atomicOr((unsigned int *)&w.ctl[CTL_ERROR], POOL_ERR_CUT_COORDS);
            }
            uint32_t tile = (uint32_t)s.cut_state[s.n_cut_state - 1][0] & 0xFF, bit = 1u << (tile & 31);
            if (!(s.cut_tiles_bits[tile >> 5] & bit)) {
                s.cut_tiles_bits[tile >> 5] |= bit;
                s.n_cut_tiles++;
            }
        }
        if (RBIT(m, 0xD803, 0)) {  // :1527-1538
            uint32_t cf13 = RAM(m, 0xCF13), ff8c = RAM(m, 0xFF8C), cf94 = RAM(m, 0xCF94);
            if (cf13 == 0 && ff8c == 6 && cf94 == 0) s.seen_start_menu = 1;
            if (cf13 == 0 && ff8c == 6 && cf94 == 2) s.seen_pokemon_menu = 1;
            if (cf13 == 0) s.seen_stats_menu = 1;
            if (cf13 == 0 && cf94 == 3) s.seen_bag_menu = 1;
        }
    }
    // :1541 update_pokedex :552-558
    int n_seen = 0, n_caught = 0;
    for (uint32_t i = 0; i < 19; i++) {
        n_caught += __popc(RAM(m, 0xD2F7 + i));
        n_seen += __popc(RAM(m, 0xD30A + i));
    }
    // :1542 update_moves_obtained :560-580
    for (uint32_t k = 0; k < 6; k++) {
        uint32_t base = 0xD16B + 44 * k;
        if (RAM(m, base) != 0)
            for (uint32_t j = 0; j < 4; j++) {
                uint32_t mv = RAM(m, base + j + 8);
                if (mv != 0) {
                    if (mv < 0xA5) s.moves_bits[mv >> 5] |= 1u << (mv & 31);
                    if (mv == 15) s.cut = 1;
                }
            }
    }
    uint32_t box_n = RAM(m, 0xDA80);
    for (uint32_t i = 0; i < box_n; i++) {
        uint32_t off = i * 200 + 0xDA96;
        if (off + 11 > 0xFFFF) break;  // the reference would raise past the address space
        if (RAM(m, off) != 0)
            for (uint32_t j = 0; j < 4; j++) {
                uint32_t mv = RAM(m, off + j + 8);
                if (mv != 0 && mv < 0xA5) s.moves_bits[mv >> 5] |= 1u << (mv & 31);
            }
    }
    int n_moves = 0;
    for (int i = 0; i < 6; i++) n_moves += __popc(s.moves_bits[i]);
    // :1544 bill_capt ram_map.py:1889-1898
    uint32_t d7f2 = RAM(m, 0xD7F2), d803 = RAM(m, 0xD803);
    int bill_capt_rew = 5 * (int)(RBIT(m, 0xD7F1, 0) + __popc(d7f2 & 0xF8) + __popc(d803 & 0x03));
    // :1547-1552
    if (RAM(m, 0xCD4D) == 61) {
        bus_write(m, 0xCD4D, 0);
        s.used_cut += 1;
    }
    // :1554-1600 reward: float64, same association order as the Python expression
    const double S = s.reward_scale;
    double start_menu = s.seen_start_menu * 0.01, pokemon_menu = s.seen_pokemon_menu * 0.1;
    double stats_menu = s.seen_stats_menu * 0.1, bag_menu = s.seen_bag_menu * 0.1;
    double cut_coords = 0.0;
    for (int i = 0; i < s.n_cut_coords; i++) cut_coords += s.cut_coords[i].value;
    cut_coords = cut_coords * 1.0;
    double cut_tiles = s.n_cut_tiles * 1.0;
    double that_guy = ((start_menu + pokemon_menu) + stats_menu) + bag_menu;
    double acc = (double)(s.max_events + bill_capt_rew);
    acc += S * (double)n_seen;
    acc += S * (double)n_caught;
    acc += S * (double)n_moves;
    acc += (double)(5 * bill_state);
    acc += (double)(hm_count * 10);
    acc += level_reward;
    acc += 0.0;
    acc += (double)(10 * badges);
    acc += s.total_healing;
    acc += exploration_reward;
    acc += (double)cut_rew;
    acc += that_guy / 2;
    acc += cut_coords;
    acc += cut_tiles;
    acc += tree_distance_reward * 0.6;
    acc += (double)(dojo_reward * 5);
    for (int k = 0; k < 5; k++) acc += s.item_reward[k];
    acc += (double)(dojo_ev + silph_ev + hideout_ev + tower_ev + g3 + g4 + g5 + g6 + g7);
    acc += (double)(g3 + g4 + g5 + g6 + g7);
    double reward_abs = S * acc, reward;
    if (!s.have_last_reward) {  // :1604-1610
        reward = 0.0;
        s.last_reward = 0.0;
        s.have_last_reward = 1;
    } else {
        reward = reward_abs - s.last_reward;
        s.last_reward = reward_abs;
    }
    s.last_delta = reward;
    *done = s.time >= s.max_episode_steps;  // :1613
    if (out) {
        out->r = r; out->c = c; out->map_n = map_n; out->party_size = party_size; out->level_sum = level_sum; out->max_level = max_level;
        out->badges = badges; out->bill_state = bill_state; out->hm_count = hm_count; out->events = events; out->money = money;
        out->n_seen = n_seen; out->n_caught = n_caught; out->n_moves = n_moves; out->dojo_reward = dojo_reward; out->bill_capt_rew = bill_capt_rew;
        out->cut_rew = cut_rew; out->level_reward = level_reward; out->exploration_reward = exploration_reward;
        out->tree_distance_reward = tree_distance_reward; out->cut_coords = cut_coords; out->cut_tiles = cut_tiles; out->start_menu = start_menu;
        out->pokemon_menu = pokemon_menu; out->stats_menu = stats_menu; out->bag_menu = bag_menu; out->reward = reward; out->reward_abs = reward_abs;
    }
    return reward;
}

// ------------------------------------------------------------------------------------- kernels

// one thread per env; grid covers the tiles.  info_rows (optional) receives the info scalars of this step.
// `skip` (may be null): envs with skip[e] != 0 do not take this step at all (gbenv_step_masked): reward 0, done 0, state and
// info row untouched
__global__ void __launch_bounds__(128) k_wrap_step(DevArrays d, WrapArrays w, double *reward, uint8_t *done, double *info_rows, const uint8_t *skip) {
    const int tile = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, env = tile * GB_TILE + lane;
    if (tile >= d.n_tiles || env >= d.n_envs) return;
    if (skip && skip[env]) {
        reward[env] = 0.0;
        done[env] = 0;
        return;
    }
    Machine m;
    machine_load(m, d, tile, lane);
    WrapState &s = w.state[env];
    int dn = 0;
    StepScalars sc;
    double rew = wrap_after_emulation(w, s, m, env, &dn, &sc);
    wrap_mark_render(w, s, m, env, false);  // render() :1812
    reward[env] = rew;
    done[env] = (uint8_t)dn;
    if (info_rows) {
        double *I = info_rows + (size_t)env * GBENV_INFO_SCALARS;
        for (int k = 0; k < GBENV_INFO_SCALARS; k++) I[k] = 0.0;
        I[GBI_COUNT] = 1; I[GBI_STEP] = s.time; I[GBI_X] = sc.c; I[GBI_Y] = sc.r; I[GBI_MAP] = sc.map_n; I[GBI_PCOUNT] = sc.party_size;
        for (uint32_t k = 0; k < 6; k++) I[GBI_LEVEL0 + k] = RAM(m, 0xD18C + 44 * k);
        I[GBI_LEVELS_SUM] = sc.level_sum; I[GBI_COORD_SUM] = (double)s.coord_sum;
        I[GBI_DEATHS] = s.death_count; I[GBI_BADGES] = sc.badges; I[GBI_OPPONENT_LEVEL] = s.max_opponent_level;
        I[GBI_MET_BILL] = RBIT(m, 0xD7F1, 0); I[GBI_USED_CELL_SEPARATOR] = RBIT(m, 0xD7F2, 3); I[GBI_SS_TICKET] = RBIT(m, 0xD7F2, 4);
        I[GBI_MET_BILL_2] = RBIT(m, 0xD7F2, 5); I[GBI_BILL_SAID] = RBIT(m, 0xD7F2, 6); I[GBI_LEFT_BILLS_HOUSE] = RBIT(m, 0xD7F2, 7);
        I[GBI_GOT_HM01] = RBIT(m, 0xD803, 0); I[GBI_RUBBED_CAPTAINS_BACK] = RBIT(m, 0xD803, 1);
        I[GBI_MAPS_EXPLORED] = s.n_seen_maps; I[GBI_PARTY_SIZE] = sc.party_size; I[GBI_HIGHEST_LEVEL] = sc.max_level;
        I[GBI_TOTAL_PARTY_LEVEL] = sc.level_sum; I[GBI_EVENT] = sc.events; I[GBI_MONEY] = sc.money; I[GBI_SEEN_POKEMON] = sc.n_seen;
        I[GBI_CAUGHT_POKEMON] = sc.n_caught; I[GBI_MOVES_OBTAINED] = sc.n_moves; I[GBI_BILL_SAVED] = sc.bill_state; I[GBI_HM_COUNT] = sc.hm_count;
        I[GBI_CUT_TAUGHT] = s.cut; I[GBI_BILL_CAPT] = sc.bill_capt_rew / 5.0; I[GBI_CUT_COORDS] = sc.cut_coords; I[GBI_CUT_TILES] = sc.cut_tiles;
        I[GBI_BAG_MENU] = sc.bag_menu; I[GBI_STATS_MENU] = sc.stats_menu; I[GBI_POKEMON_MENU] = sc.pokemon_menu; I[GBI_START_MENU] = sc.start_menu;
        I[GBI_USED_CUT] = s.used_cut; I[GBI_DEFEATED_DOJO] = RBIT(m, 0xD7B1, 0); I[GBI_GOT_HITMONLEE] = 3 * RBIT(m, 0xD7B1, 6);
        I[GBI_GOT_HITMONCHAN] = 3 * RBIT(m, 0xD7B1, 7);
        I[GBI_R_DELTA] = sc.reward; I[GBI_R_EVENT] = s.max_events; I[GBI_R_LEVEL] = sc.level_reward;
        I[GBI_R_OPPONENT_LEVEL] = 0.006 * s.max_opponent_level; I[GBI_R_BADGES] = 10 * sc.badges; I[GBI_R_BILL_SAVED] = 5 * sc.bill_state;
        I[GBI_R_HM_COUNT] = sc.hm_count * 10; I[GBI_R_HEALING] = s.total_healing; I[GBI_R_EXPLORATION] = sc.exploration_reward;
        I[GBI_R_TREE_DISTANCE] = sc.tree_distance_reward; I[GBI_R_DOJO_OLD] = sc.dojo_reward;
        I[GBI_R_ITEMS] = s.item_reward[0] + s.item_reward[1] + s.item_reward[2] + s.item_reward[3] + s.item_reward[4];
        I[GBI_R_USED_CUT] = sc.cut_rew; I[GBI_R_ABS] = sc.reward_abs; I[GBI_SEEN_COORDS] = s.n_seen_coords; I[GBI_DONE] = dn;
        for (int k = 0; k < 5; k++) I[GBI_R_LEMONADE + k] = s.item_reward[k];
    }
    // the wrapper only writes plain WRAM bytes (straight to HBM): no register write-back is needed
}

// Environment.reset wrapper half for masked envs (state load is done by k_scatter_image beforehand)
__global__ void k_wrap_reset_pre(DevArrays d, WrapArrays w, const uint8_t *mask) {
    // :1239 get_base_event_flags: mem[D778] |= 0x10 happens BEFORE the (first-reset-only) state load
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= d.n_envs || (mask && !mask[env])) return;
    Machine m;
    machine_load(m, d, env >> 5, env & 31);
    bus_write(m, 0xD778, RAM(m, 0xD778) | 0x10);
}

__global__ void k_wrap_reset_post(DevArrays d, WrapArrays w, const uint8_t *mask, int max_episode_steps, double reward_scale) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= d.n_envs || (mask && !mask[env])) return;
    WrapState &s = w.state[env];
    Machine m;
    machine_load(m, d, env >> 5, env & 31);
    // screen_memory / seen_coords are rebuilt (:1251-1266): k_vis_release has returned this env's bitmap pages to the pool
    s.reset_count += 1;
    s.time = 0;
    s.max_episode_steps = max_episode_steps;
    s.reward_scale = reward_scale;
    s.have_last_reward = 0;
    s.last_reward = 0.0;
    s.last_delta = 0.0;
    s.prev_map_n = -2;
    s.max_events = 0; s.max_level_sum = 0; s.max_opponent_level = 0;
    s.n_seen_coords = 0; s.n_seen_maps = 0;
    for (int k = 0; k < 8; k++) { s.seen_maps_bits[k] = 0; s.cut_tiles_bits[k] = 0; }
    for (int k = 0; k < 6; k++) s.moves_bits[k] = 0;
    s.death_count = 0;
    s.total_healing = 0.0;
    s.last_hp = 1.0;
    s.last_party_size = 1;
    s.hm_latch = 0; s.cut = 0; s.used_cut = 0;
    s.n_cut_coords = 0; s.n_cut_tiles = 0; s.n_cut_state = 0;
    s.seen_start_menu = s.seen_pokemon_menu = s.seen_stats_menu = s.seen_bag_menu = 0;
    s.last_map_id_plus1 = 0;
    s.reset_pending = 0;
    update_last_map_id(m, s);              // :1327
    wrap_mark_render(w, s, m, env, true);  // :1334 render()
}

__global__ void k_wrap_init(WrapArrays w, int n_envs) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= n_envs) return;
    WrapState &s = w.state[env];
    // state memory was zero-filled by the host; set the non-zero defaults of Environment.__init__
    s.last_map = -1;
    s.initial_template = -1;
    s.prev_map_n = -2;
    s.last_hp = 1.0;
    s.last_party_size = 1;
    s.reward_scale = 1.0;
    s.max_episode_steps = 20480;
}

// Reset, first half of the exploration storage: the visited-bitmap pages of every masked env go back to the free stack,
// zeroed.  One block per env; runs before k_wrap_reset_post (which pops a page for the tile render() marks), so pushes and
// pops never meet in one launch.
__global__ void __launch_bounds__(256) k_vis_release(WrapArrays w, const uint8_t *mask, int n_envs) {
    const int env = blockIdx.x;
    if (env >= n_envs || (mask && !mask[env])) return;
    uint32_t *pt = w.vis_pt + (size_t)env * VIS_PT_ENTRIES;
    for (int k = threadIdx.x; k < VIS_PT_ENTRIES; k += blockDim.x) {
        const uint32_t pg = pt[k];
        if (!pg) continue;
        uint4 *page = (uint4 *)(w.vis_pool + (size_t)(pg - 1) * VIS_PAGE_WORDS);
        for (int i = 0; i < VIS_PAGE_WORDS / 4; i++) page[i] = make_uint4(0, 0, 0, 0);
        pt[k] = 0;
        w.vis_free[atomicAdd(&w.ctl[CTL_VIS_FREE], 1)] = (int32_t)(pg - 1);
    }
}

// gbenv_counts_map: one env's heat map as the dense 444 x 436 image; one block per heat-map block
__global__ void __launch_bounds__(CM_BLOCK * CM_BLOCK) k_cm_gather(WrapArrays w, int env, int32_t *dense) {
    const int by = blockIdx.x / CM_BLOCKS_X, bx = blockIdx.x % CM_BLOCKS_X, y = by * CM_BLOCK + threadIdx.x / CM_BLOCK, x = bx * CM_BLOCK + threadIdx.x % CM_BLOCK;
    if (y >= COUNTS_H || x >= COUNTS_W) return;
    const uint32_t b = w.cm_dir[(size_t)env * CM_DIR_ENTRIES + blockIdx.x];
    dense[y * COUNTS_W + x] = b ? w.cm_pool[(size_t)(b - 1) * (CM_BLOCK * CM_BLOCK) + threadIdx.x] : 0;
}

// gbenv_counts_map_sum: sum[cell] += the cell over the heat maps of the envs [chunk * chunk_envs, +chunk_envs) with mask[e] != 0
// (mask null: all).  grid (CM_DIR_ENTRIES, chunks), CM_SUM_THREADS threads; sum is zeroed beforehand on the same stream.
// Envs that start from one save-state walk the same cells, so a per-(env, cell) atomic would pile onto a few addresses.  Instead
// each warp takes CM_SUM_GROUP envs at a time: a lane reads the directory entries and mask bytes of CM_SUM_GROUP / 32 envs (all
// loads in flight together), a ballot per 32 envs names the lanes with a present, masked block, and the warp then reads those
// blocks whole (1 KiB, two 16-byte loads per lane) into 8 int64 partial sums per lane (cells 4l..4l+3 and 128+4l..128+4l+3).
// The warps' partials meet in shared memory; each cell then takes one 64-bit atomicAdd per block.  Integer sums: the result
// does not depend on the order in which blocks run.
#define CM_SUM_THREADS 256
#define CM_SUM_GROUP 128
__global__ void __launch_bounds__(CM_SUM_THREADS) k_cm_sum(WrapArrays w, const uint8_t *mask, int n_envs, int chunk_envs, long long *sum) {
    __shared__ long long s_part[CM_SUM_THREADS / 32][CM_BLOCK * CM_BLOCK];
    const int entry = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e_begin = blockIdx.y * chunk_envs, e_end = min(n_envs, e_begin + chunk_envs);
    long long acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int base = e_begin + warp * CM_SUM_GROUP; base < e_end; base += CM_SUM_GROUP * (CM_SUM_THREADS / 32)) {
        uint32_t dir[CM_SUM_GROUP / 32];
#pragma unroll
        for (int u = 0; u < CM_SUM_GROUP / 32; u++) {
            const int e = base + u * 32 + lane;
            dir[u] = (e < e_end && (!mask || mask[e])) ? w.cm_dir[(size_t)e * CM_DIR_ENTRIES + entry] : 0u;
        }
#pragma unroll
        for (int u = 0; u < CM_SUM_GROUP / 32; u++) {
            uint32_t bits = __ballot_sync(0xFFFFFFFFu, dir[u] != 0);
            while (bits) {  // two blocks per pass, so that four 16-byte loads per lane are in flight
                const int l0 = __ffs(bits) - 1;
                bits &= bits - 1;
                const int l1 = bits ? __ffs(bits) - 1 : l0;
                const bool two = bits != 0;
                bits &= bits - 1;
                const uint32_t b0 = __shfl_sync(0xFFFFFFFFu, dir[u], l0), b1 = __shfl_sync(0xFFFFFFFFu, dir[u], l1);
                const int4 *p0 = (const int4 *)(w.cm_pool + (size_t)(b0 - 1) * (CM_BLOCK * CM_BLOCK)) + lane;
                const int4 *p1 = (const int4 *)(w.cm_pool + (size_t)(b1 - 1) * (CM_BLOCK * CM_BLOCK)) + lane;
                const int4 a0 = p0[0], a1 = p0[32];
                int4 c0 = make_int4(0, 0, 0, 0), c1 = c0;
                if (two) { c0 = p1[0]; c1 = p1[32]; }
                acc[0] += (long long)a0.x + c0.x; acc[1] += (long long)a0.y + c0.y; acc[2] += (long long)a0.z + c0.z; acc[3] += (long long)a0.w + c0.w;
                acc[4] += (long long)a1.x + c1.x; acc[5] += (long long)a1.y + c1.y; acc[6] += (long long)a1.z + c1.z; acc[7] += (long long)a1.w + c1.w;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        s_part[warp][4 * lane + k] = acc[k];
        s_part[warp][128 + 4 * lane + k] = acc[4 + k];
    }
    __syncthreads();
    const int cell = threadIdx.x, by = entry / CM_BLOCKS_X, bx = entry % CM_BLOCKS_X;
    const int y = by * CM_BLOCK + cell / CM_BLOCK, x = bx * CM_BLOCK + cell % CM_BLOCK;
    long long t = 0;
#pragma unroll
    for (int k = 0; k < CM_SUM_THREADS / 32; k++) t += s_part[k][cell];
    if (t != 0 && y < COUNTS_H && x < COUNTS_W) atomicAdd((unsigned long long *)&sum[y * COUNTS_W + x], (unsigned long long)t);
}

// Observation assembly: block = one 32-env tile, 256 threads.  For each of the 72 output rows the block
// loads the even framebuffer line (10 words x 32 lanes, coalesced), then writes 32 x 80 RGBA-like pixels
// as 32-bit words: [grey, grey, grey, visited] (environment.py:266-272, :233-254).
// `mask` (may be null) selects the envs whose rows are written: mask[e] != 0, or mask[e] == 0 when `invert` is set
__global__ void __launch_bounds__(256) k_wrap_obs(DevArrays d, WrapArrays w, const uint8_t *mask, uint8_t *obs, size_t obs_stride, int invert = 0) {
    __shared__ uint32_t s_fb[FB_LINE_WORDS][32];
    __shared__ uint32_t s_win[32][3];  // 80-bit visited window of the current row, per env
    __shared__ int s_r[32], s_c[32];
    __shared__ uint32_t s_page[32][VIS_BANDS];  // the current map's bitmap pages (index + 1, 0 = none)
    const int tile = blockIdx.x, tid = threadIdx.x;
    if (tid < 32) {
        int env = tile * 32 + tid;
        int r = 0, c = 0;
        for (int b = 0; b < VIS_BANDS; b++) s_page[tid][b] = 0;
        if (env < d.n_envs) {
            const uint8_t *memb = (const uint8_t *)(d.mem + il_index(tile, MEM_WORDS, 0, tid));
            auto rd = [&](uint32_t a) { uint32_t i = MEM_WRAM + (a - 0xC000); return (int)memb[((i >> 2) << 7) | (i & 3)]; };
            r = rd(0xD361);
            c = rd(0xD362);
            int map_n = rd(0xD35E);
            map_n = map_n > 247 ? 247 : map_n;
            for (int b = 0; b < VIS_BANDS; b++) s_page[tid][b] = w.vis_pt[(size_t)env * VIS_PT_ENTRIES + map_n * VIS_BANDS + b];
        }
        s_r[tid] = r; s_c[tid] = c;
    }
    __syncthreads();
    const uint32_t grey_lut = 0x00559900u | 0xFFu;  // shade 0..3 -> 0xFF 0x99 0x55 0x00 (byte k of the word)
    for (int i = 0; i < 72; i++) {
        for (int k = tid; k < FB_LINE_WORDS * 32; k += 256) {
            int wd = k >> 5, lane = k & 31;
            s_fb[wd][lane] = d.fb[il_index(tile, FB_WORDS, (uint32_t)(2 * i) * FB_LINE_WORDS + wd, lane)];
        }
        if (tid < 96) {  // visited window: columns c-40 .. c+39 of bitmap row r-36+i
            int e = tid / 3, part = tid % 3, env = tile * 32 + e;
            uint32_t bits = 0;
            int rr = s_r[e] - 36 + i;
            const uint32_t pg = (env < d.n_envs && rr >= 0 && rr < 255) ? s_page[e][rr / VIS_BAND_ROWS] : 0;
            if (pg) {
                const uint32_t *row = w.vis_pool + (size_t)(pg - 1) * VIS_PAGE_WORDS + (rr % VIS_BAND_ROWS) * VIS_ROW_WORDS;
                int c0 = s_c[e] - 40 + part * 32;  // first column of this 32-bit part
                for (int b = 0; b < 32; b++) {
                    int cc = c0 + b;
                    if (cc >= 0 && cc < 255 && part * 32 + b < 80) bits |= ((row[cc >> 5] >> (cc & 31)) & 1u) << b;
                }
            }
            s_win[e][part] = bits;
        }
        __syncthreads();
        for (int k = tid; k < 32 * 80; k += 256) {
            int e = k / 80, j = k % 80, env = tile * 32 + e;
            if (env < d.n_envs && (!mask || (mask[env] != 0) != (invert != 0))) {
                uint32_t shade = (s_fb[j >> 3][e] >> (4 * (j & 7))) & 3;  // pixel x = 2j
                uint32_t g = (grey_lut >> (8 * shade)) & 0xFF;
                uint32_t vis = (s_win[e][j >> 5] >> (j & 31)) & 1 ? 0xFFu : 0u;
                uint32_t px = g | (g << 8) | (g << 16) | (vis << 24);
                *(uint32_t *)(obs + (size_t)env * obs_stride + (size_t)(i * 80 + j) * 4) = px;
            }
        }
        __syncthreads();
    }
}

// sum of the info rows over the envs with mask[e] != 0 (mask null: all) -> GBENV_INFO_SCALARS doubles (the vector multi-GPU
// runs all-reduce over NCCL).  A masked-out row is skipped, so the unmasked envs are added in the same order as without a mask.
__global__ void k_reduce_info(const double *rows, const uint8_t *mask, int n_envs, double *sum) {
    __shared__ double s[256];
    const int k = blockIdx.x;  // one block per info slot
    double acc = 0.0;
    for (int e = threadIdx.x; e < n_envs; e += blockDim.x)
        if (!mask || mask[e]) acc += rows[(size_t)e * GBENV_INFO_SCALARS + k];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int st = blockDim.x / 2; st > 0; st >>= 1) {
        if (threadIdx.x < st) s[threadIdx.x] += s[threadIdx.x + st];
        __syncthreads();
    }
    if (threadIdx.x == 0) sum[k] = s[0];
}
