"""Names of the per-env info row (include/gbenv_info.h) and its conversion to the reference's info dict
layout (`info["stats"]`, `info["reward"]`; /root/reference/pokegym/environment.py:1621-1703)."""
from __future__ import annotations

import json
import re
from pathlib import Path
from typing import Callable, Dict, List, Optional

import numpy as np


def names_from_header(path=None) -> List[str]:
    """The same list parsed from include/gbenv_info.h (source checkouts only: the test that keeps _info_names.py in step)."""
    text = Path(path or Path(__file__).resolve().parent.parent / "include" / "gbenv_info.h").read_text()
    body = text[text.index("enum {") : text.index("GBI__END")]
    names: List[str] = []
    for tok in re.findall(r"GBI_([A-Z0-9_]+)(?:\s*=\s*([^,]+))?,", body):
        name, init = tok
        if name == "LEVEL0":
            names += [f"level{k}" for k in range(6)]
        elif name == "LEVELS_SUM" and init:
            names.append("levels_sum")
        elif name != "COUNT" or not names:
            names.append(name.lower())
    return names


from ._info_names import INFO_NAMES  # noqa: E402  (generated from include/gbenv_info.h)

INFO_INDEX: Dict[str, int] = {n: i for i, n in enumerate(INFO_NAMES)}
assert len(INFO_NAMES) <= 72 and INFO_NAMES[0] == "count", INFO_NAMES[:3]

_REWARD_KEYS = {"r_delta": "delta", "r_event": "event", "r_level": "level", "r_opponent_level": "opponent_level", "r_badges": "badges",
                "r_bill_saved": "bill_saved_reward", "r_hm_count": "hm_count_reward", "r_healing": "healing", "r_exploration": "exploration",
                "r_tree_distance": "tree_distance_reward", "r_dojo_old": "dojo_reward_old", "r_used_cut": "used_cut_reward"}


def info_row_to_dict(row: np.ndarray) -> dict:
    """One info row -> {"stats": {...}, "reward": {...}} with the reference's key names where they exist."""
    stats, reward = {}, {}
    for i, name in enumerate(INFO_NAMES):
        v = float(row[i])
        if name in _REWARD_KEYS:
            reward[_REWARD_KEYS[name]] = v
        elif name.startswith("r_"):
            reward[name[2:]] = v
        elif name not in ("count",):
            stats[name] = v
    stats["levels"] = [stats.pop(f"level{k}") for k in range(6)]
    for k in range(1, 7):
        stats[f"badge_{k}"] = float(stats["badges"] >= k)
    return {"stats": stats, "reward": reward}


def info_sum_to_means(total: np.ndarray) -> Dict[str, float]:
    """All-reduced sum vector -> per-env means (slot 0 carries the env count)."""
    n = max(float(total[0]), 1.0)
    return {name: float(total[i]) / n for i, name in enumerate(INFO_NAMES) if name != "count"}


# ---------------------------------------------------------------------------------------------------
# Full info dict (environment.py:1621-1810): the scalar row + the 130 named event bits + counts_map.

_GROUPS = ("silph_co", "dojo", "hideout", "poke_tower", "gym3", "gym4", "gym5", "gym6", "gym7")
_EVENT_TABLE: Optional[Dict[str, list]] = None


def event_table() -> Dict[str, list]:
    """group -> [[name, address, bit, weight], ...] in the reference's dict order (ram_map_leanke.py:107-164, 816-827,
    867-889, 936-957, 1038-1098).  Data file written by tools/gen_reference_tables.py; same bits as c_events in gb_wrap.cuh."""
    global _EVENT_TABLE
    if _EVENT_TABLE is None:
        _EVENT_TABLE = json.loads((Path(__file__).resolve().parent / "event_table.json").read_text())
        assert tuple(_EVENT_TABLE) == _GROUPS and sum(len(v) for v in _EVENT_TABLE.values()) == 130
    return _EVENT_TABLE


def event_rewards_detailed(events: Dict[str, int], base_reward=10, reward_increment=2, reward_multiplier=1) -> Dict[str, int]:
    """environment.py:1221-1231: base + value*increment*multiplier for positive entries, value*increment*multiplier otherwise."""
    return {k: (base_reward if v > 0 else 0) + v * reward_increment * reward_multiplier for k, v in events.items()}


def event_bits(read_byte: Callable[[int], int]) -> np.ndarray:
    """uint8 [130]: the bit that entry k of the event table reads (`read_byte(addr)`, e.g. gbenv_read_mem), in table order
    (silph_co, dojo, hideout, poke_tower, gym3..gym7), whatever the sign of its weight."""
    return np.array([(read_byte(a) >> b) & 1 for g in _GROUPS for _, a, b, _ in event_table()[g]], dtype=np.uint8)


def unpack_event_words(words) -> np.ndarray:
    """gbenv_event_flags rows [n, 5] (uint32 or int32 words: bit k & 31 of word k >> 5 is entry k) -> uint8 [n, 130]."""
    if hasattr(words, "detach"):
        words = words.detach().cpu().numpy()
    w = np.ascontiguousarray(words)
    if w.ndim != 2 or w.shape[1] != 5 or w.dtype.itemsize != 4:
        raise ValueError("event words must be a [n, 5] array of 32-bit words")
    return np.unpackbits(w.astype("<u4", copy=False).view(np.uint8), axis=1, bitorder="little")[:, :130]


def _event_entries(ev: Dict[str, dict], detailed: Dict[str, dict]) -> dict:
    """The event part of the info dict (environment.py:1790-1810) from per-group {name: value} dicts."""
    return {
        "detailed_rewards_silph_co": detailed["silph_co"], "detailed_rewards_dojo": detailed["dojo"],
        "detailed_rewards_hideout": detailed["hideout"], "detailed_rewards_poke_tower": detailed["poke_tower"],
        "detailed_rewards_gyms": {f"gym_{k}_detailed_rewards": detailed[f"gym{k}"] for k in range(3, 8)},
        "silph_co_events_aggregate": ev["silph_co"], "dojo_events_aggregate": ev["dojo"], "hideout_events_aggregate": ev["hideout"],
        "poke_tower_events_aggregate": ev["poke_tower"], "gym_events": {f"gym_{k}_events": ev[f"gym{k}"] for k in range(3, 8)},
    }


def _by_group(values) -> Dict[str, list]:
    """group -> [(name, weight, value of its entry)] for one value per table entry, in table order."""
    out, k = {}, 0
    for g in _GROUPS:
        out[g] = [(name, w, values[k + j]) for j, (name, _, _, w) in enumerate(event_table()[g])]
        k += len(out[g])
    return out


def event_counts_to_means(counts, n) -> dict:
    """Counts of set event flags over n envs (int64 [130], e.g. VecEnvironment.event_counts, all-reduced or not) -> the
    nine aggregate dicts and the `detailed_rewards_*` dicts as means over those n envs, under the reference's keys.  Per env
    an aggregate entry is weight * bit and a detailed one (10 if weight * bit > 0 else 0) + 2 * weight * bit."""
    if hasattr(counts, "detach"):
        counts = counts.detach().cpu().numpy()
    c = np.asarray(counts, dtype=np.float64).reshape(-1)
    if c.size != 130:
        raise ValueError("counts must have 130 entries")
    n = max(float(n), 1.0)
    groups = _by_group(c)
    ev = {g: {name: w * v / n for name, w, v in rows} for g, rows in groups.items()}
    detailed = {g: {name: ((10 if w > 0 else 0) + 2 * w) * v / n for name, w, v in rows} for g, rows in groups.items()}
    return _event_entries(ev, detailed)


def build_info(row: np.ndarray, read_byte: Callable[[int], int], counts_map: Optional[np.ndarray] = None, reward_scale: float = 4.0) -> dict:
    """The dict `Environment.step` returns when `done or time % 10000 == 0` (environment.py:1621-1810), rebuilt from one
    info row, the env's event bytes (`read_byte(addr)`, e.g. gbenv_read_mem) and its counts_map."""
    return build_info_from_events(row, event_bits(read_byte), counts_map=counts_map, reward_scale=reward_scale)


def build_info_from_events(row: np.ndarray, bits, counts_map: Optional[np.ndarray] = None, reward_scale: float = 4.0) -> dict:
    """build_info from one info row, the env's 130 event bits (event_bits, or a row of unpack_event_words) and its
    counts_map.

    Entries the reference fills from state it never updates are emitted with the constant it would hold
    (`self.badge_count`, `events`, `seen_npcs_count`, `hidden_obj_count`, `state_loaded_instead_of_resetting_in_game`: 0).
    `maps_explored` is the number of distinct maps seen (the reference's later duplicate key stores the raw set object)."""
    I = {n: float(row[i]) for i, n in enumerate(INFO_NAMES)}
    levels = [int(I[f"level{k}"]) for k in range(6)]
    badges = I["badges"]
    stats = {
        "step": int(I["step"]), "x": int(I["x"]), "y": int(I["y"]), "map": int(I["map"]), "pcount": int(I["pcount"]), "levels": levels,
        "levels_sum": int(I["levels_sum"]), "coord": I["coord_sum"], "deaths": int(I["deaths"]), "deaths_per_episode": int(I["deaths"]),
        "badges": badges, "self.badge_count": 0, **{f"badge_{k}": float(badges >= k) for k in range(1, 7)}, "events": 0,
        "opponent_level": int(I["opponent_level"]), "met_bill": int(I["met_bill"]), "used_cell_separator_on_bill": int(I["used_cell_separator"]),
        "ss_ticket": int(I["ss_ticket"]), "met_bill_2": int(I["met_bill_2"]), "bill_said_use_cell_separator": int(I["bill_said"]),
        "left_bills_house_after_helping": int(I["left_bills_house"]), "got_hm01": int(I["got_hm01"]),
        "rubbed_captains_back": int(I["rubbed_captains_back"]), "maps_explored": int(I["maps_explored"]), "party_size": int(I["party_size"]),
        "highest_pokemon_level": int(I["highest_level"]), "total_party_level": int(I["total_party_level"]), "event": int(I["event"]),
        "money": int(I["money"]), "pokemon_exploration_map": counts_map, "seen_npcs_count": 0, "seen_pokemon": I["seen_pokemon"],
        "caught_pokemon": I["caught_pokemon"], "moves_obtained": I["moves_obtained"], "hidden_obj_count": 0, "bill_saved": int(I["bill_saved"]),
        "hm_count": int(I["hm_count"]), "cut_taught": int(I["cut_taught"]), "bill_capt": I["bill_capt"], "cut_coords": I["cut_coords"],
        "cut_tiles": I["cut_tiles"], "bag_menu": I["bag_menu"], "stats_menu": I["stats_menu"], "pokemon_menu": I["pokemon_menu"],
        "start_menu": I["start_menu"], "used_cut": int(I["used_cut"]), "state_loaded_instead_of_resetting_in_game": 0,
        "defeated_fighting_dojo": int(I["defeated_dojo"]), "got_hitmonlee": int(I["got_hitmonlee"]), "got_hitmonchan": int(I["got_hitmonchan"]),
    }
    reward = {
        "delta": I["r_delta"], "event": I["r_event"], "level": I["r_level"], "opponent_level": I["r_opponent_level"], "death": 0,
        "badges": I["r_badges"], "bill_saved_reward": I["r_bill_saved"], "hm_count_reward": I["r_hm_count"], "healing": I["r_healing"],
        "exploration": I["r_exploration"], "seen_pokemon_reward": reward_scale * I["seen_pokemon"],
        "caught_pokemon_reward": reward_scale * I["caught_pokemon"], "moves_obtained_reward": reward_scale * I["moves_obtained"],
        "used_cut_reward": I["r_used_cut"], "tree_distance_reward": I["r_tree_distance"], "dojo_reward_old": I["r_dojo_old"],
        "has_lemonade_in_bag_reward": I["r_lemonade"], "has_silph_scope_in_bag_reward": I["r_silph_scope"],
        "has_lift_key_in_bag_reward": I["r_lift_key"], "has_pokedoll_in_bag_reward": I["r_pokedoll"], "has_bicycle_in_bag_reward": I["r_bicycle"],
    }
    ev = {g: {name: w * int(b) for name, w, b in rows} for g, rows in _by_group(bits).items()}  # monitor_<group>_events
    return {"pokemon_exploration_map": counts_map, "stats": stats, "reward": reward,
            **_event_entries(ev, {g: event_rewards_detailed(v) for g, v in ev.items()})}
