"""CPU suite: the oracle against the committed golden vectors (no GPU, no /root/reference needed)."""
import numpy as np
import pytest

from helpers import GOLDEN, check_ppu_kat, load_wrapper_sweep, replay_wrapper_golden, replay_wrapper_sweep
from pokegym_b200 import _capi


@pytest.mark.parametrize("name", ["pokelike_a", "pokelike_b", "red_overworld", "red_battle", "red_bill", "red_pallet"])
def test_oracle_replays_reference_wrapper_recording(oracle_lib, roms, name):
    gold = np.load(GOLDEN / f"ref_wrapper_{name}.npz")
    h = _capi.Handle(oracle_lib, 1, roms(str(gold["rom_name"])))
    replay_wrapper_golden(h, gold)


def test_oracle_renderer_matches_pyboy_framebuffers(oracle_lib, roms):
    kat = np.load(GOLDEN / "ppu_kat.npz")
    h = _capi.Handle(oracle_lib, 1, roms("pokelike"))
    check_ppu_kat(h, kat)


def test_oracle_replays_reference_wrapper_on_all_264_states(oracle_lib, roms):
    gold = load_wrapper_sweep()
    replay_wrapper_sweep(_capi.Handle(oracle_lib, len(gold["names"]), roms("pokelike")), gold)
