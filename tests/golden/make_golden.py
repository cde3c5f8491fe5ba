#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ (run in the build container, needs /root/reference).

1. ref_wrapper_*.npz -- the UNMODIFIED reference `pokegym.Environment` stepped on the PyBoy shim
   (tests/ref_shim.py) over the oracle emulator core with the synthetic Pokemon-like ROM: per-step reward
   (float64), done, CRC32 of the (72,80,4) observation, SHA-256 of the full emulator state, the wrapper's
   RAM writes, the start state, and a fingerprint of every info dict the reference emitted.  Recorded from a booted
   synthetic game (pokelike_*) and from four of the reference's real Pokemon Red save-states (red_*).  GPU tests replay
   the same actions through the CUDA path.
2. ppu_kat.npz -- for a spread of the reference's own PyBoy save-states: the renderer inputs (VRAM, OAM,
   LCD registers, per-scanline parameters) and the framebuffer PyBoy itself rendered from them (2 bits per
   pixel).  These pin the scanline renderer to real PyBoy output.
"""
import hashlib
import json
import lzma
import sys
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import __graft_entry__ as g  # noqa: E402
from helpers import info_fingerprint  # noqa: E402
from pokegym_b200 import _capi  # noqa: E402
from pokegym_b200.state_file import parse_state  # noqa: E402
from pokegym_b200.tools import synth_rom  # noqa: E402

OUT = Path(__file__).resolve().parent
REF = Path("/root/reference/pokegym")
SHADE_OF = {0xFFFFFF01: 0, 0x99999900: 1, 0x55555500: 2, 0x00000000: 3}


def wrapper_golden(name, rom_name, start_blob, n_steps, seed, max_episode_steps, reset_at, oracle_lib):
    import ref_shim

    rom_fn, kw = synth_rom.rom_catalog()[rom_name]
    rom = rom_fn(**kw)
    rng = np.random.default_rng(seed)
    actions = rng.integers(0, 8, n_steps).astype(np.uint8)
    ref = ref_shim.run_reference_episode(rom, oracle_lib, start_blob, actions, max_episode_steps=max_episode_steps, reset_at=reset_at)
    obs_crc = np.array([zlib.crc32(o.tobytes()) for o in ref["obs"]], dtype=np.uint32)
    state_sha = np.array([np.frombuffer(hashlib.sha256(s).digest(), dtype=np.uint8) for s in ref["states"]])
    writes = np.array([len(w) for w in ref["writes"]], dtype=np.int32)
    info_steps = [i for i, x in enumerate(ref["infos"]) if x]
    info_json = [json.dumps(info_fingerprint(ref["infos"][i])) for i in info_steps]
    np.savez_compressed(
        OUT / f"ref_wrapper_{name}.npz", rom_name=rom_name, start_state=np.frombuffer(start_blob, dtype=np.uint8), actions=actions,
        rewards=np.array(ref["rewards"], dtype=np.float64), dones=np.array(ref["dones"], dtype=np.uint8), obs_crc=obs_crc, state_sha=state_sha,
        n_ram_writes=writes, max_episode_steps=max_episode_steps, reset_at=np.array(reset_at, dtype=np.int32),
        reset_obs_crc=np.array([zlib.crc32(o.tobytes()) for o in ref["reset_obs"]], dtype=np.uint32), last_obs=ref["obs"][-1],
        info_steps=np.array(info_steps, dtype=np.int32), info_json=np.array(info_json))
    print(name, "steps", n_steps, "info dicts", len(info_steps), "sum|reward|", float(np.abs(ref["rewards"]).sum()), "nonzero rewards", int(np.count_nonzero(ref["rewards"])))


def ppu_golden(n_pick=264):  # every v9 fixture the reference ships
    files = sorted(p for p in REF.rglob("*") if p.is_file() and p.stat().st_size == 142_610)
    # spread over the fixture directories; prefer states with a visible window / many sprites
    pick = [files[i] for i in np.linspace(0, len(files) - 1, n_pick).astype(int)]
    recs = dict(vram=[], oam=[], lcd_regs=[], scanline_params=[], fb2=[], names=[])
    for p in pick:
        st = parse_state(p.read_bytes())
        words = np.frombuffer(st.raw["screen"].tobytes(), dtype="<u4")
        shades = np.vectorize(SHADE_OF.__getitem__, otypes=[np.uint8])(words)
        recs["vram"].append(st.raw["vram"])
        recs["oam"].append(st.raw["oam"])
        recs["lcd_regs"].append(st.raw["lcd_regs"])
        recs["scanline_params"].append(st.raw["scanline_params"])
        recs["fb2"].append(np.packbits(np.unpackbits(shades[:, None], axis=1)[:, 6:].reshape(-1)))  # 2 bits per pixel
        recs["names"].append(str(p.relative_to(REF)))
    np.savez_compressed(OUT / "ppu_kat.npz", **{k: np.array(v) for k, v in recs.items()})
    print("ppu_kat:", len(pick), "fixtures")


def wrapper_sweep_golden(oracle_lib, n_steps=6):
    """3. ref_wrapper_sweep.npz -- ALL 264 v9 save-states the reference ships, each reset + stepped `n_steps` times by the
    unmodified reference wrapper (on the PyBoy shim over the oracle core, synthetic ROM): reward, done, observation CRC and
    state hash per step.  The states cover every outcome of Game.process_game_states (red_ram_api.py:59-73, :149-225,
    :542-602), wild / trainer battles, menus and overworld; one batch of 264 envs replays them through CUDA."""
    import ref_shim

    rom = synth_rom.build_pokelike_rom()
    files = sorted(p for p in REF.rglob("*") if p.is_file() and p.stat().st_size == 142_610)
    rng = np.random.default_rng(264)
    actions = rng.integers(0, 8, (len(files), n_steps)).astype(np.uint8)
    rec = dict(states=[], names=[], rewards=[], dones=[], obs_crc=[], reset_obs_crc=[], state_sha=[])
    for k, p in enumerate(files):
        blob = p.read_bytes()
        ref = ref_shim.run_reference_episode(rom, oracle_lib, blob, actions[k], max_episode_steps=4)  # done fires at step 4
        rec["states"].append(np.frombuffer(blob, dtype=np.uint8))
        rec["names"].append(str(p.relative_to(REF)))
        rec["rewards"].append(ref["rewards"])
        rec["dones"].append(ref["dones"])
        rec["obs_crc"].append([zlib.crc32(o.tobytes()) for o in ref["obs"]])
        rec["reset_obs_crc"].append(zlib.crc32(ref["reset_obs"][0].tobytes()))
        rec["state_sha"].append(np.frombuffer(hashlib.sha256(ref["states"][-1]).digest(), dtype=np.uint8))
    states_xz = np.frombuffer(lzma.compress(np.stack(rec["states"]).tobytes(), preset=9 | lzma.PRESET_EXTREME), dtype=np.uint8)  # helpers.load_wrapper_sweep
    np.savez_compressed(OUT / "ref_wrapper_sweep.npz", states_xz=states_xz, names=np.array(rec["names"]), actions=actions,
                        rewards=np.array(rec["rewards"], dtype=np.float64), dones=np.array(rec["dones"], dtype=np.uint8),
                        obs_crc=np.array(rec["obs_crc"], dtype=np.uint32), reset_obs_crc=np.array(rec["reset_obs_crc"], dtype=np.uint32),
                        state_sha=np.stack(rec["state_sha"]), max_episode_steps=4)
    print("ref_wrapper_sweep:", len(files), "states x", n_steps, "steps; distinct rewards", len(set(np.array(rec["rewards"]).ravel().tolist())))


def main():
    lib = _capi.GbEnvLib(g.build_oracle(), "oracle_")
    rom = synth_rom.build_pokelike_rom()
    h = _capi.Handle(lib, 1, rom)
    h.tick(60, True)
    start = h.save_state(0)
    wrapper_golden("pokelike_a", "pokelike", start, 400, 11, 150, (150, 300), lib)
    wrapper_golden("pokelike_b", "pokelike", start, 250, 12, 20480, (), lib)
    # real Pokemon Red RAM (party, events, bag, battle / menu state) from the reference's own save-states, driven by the
    # state-compatible synthetic ROM: pins reward shaping, RAM side effects and the info dict on game data
    for name, rel in (("red_overworld", "current_state/Bulbasaur.state"), ("red_battle", "bin/checkpoints_battles/bulbasaur/pokemon_ai_14"),
                      ("red_bill", "bin/checkpoints_bill/pokemon_ai_1005"), ("red_pallet", "bin/checkpoints_pallet/pokemon_ai_105")):
        p = REF / rel
        if not p.exists():
            cands = sorted(p.parent.glob("*"))
            p = cands[len(cands) // 2]
        wrapper_golden(name, "pokelike", p.read_bytes(), 60, 7, 40, (45,), lib)
    ppu_golden()
    wrapper_sweep_golden(lib)


if __name__ == "__main__":
    main()
