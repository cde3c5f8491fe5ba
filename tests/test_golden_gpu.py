"""GPU suite: the CUDA path against the golden vectors recorded from the reference's own wrapper and from
PyBoy's own framebuffers (run on the B200 box; /root/reference does not exist there)."""
import numpy as np
import pytest

from helpers import GOLDEN, check_ppu_kat, load_wrapper_sweep, replay_wrapper_golden, replay_wrapper_sweep
from pokegym_b200 import _capi

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["pokelike_a", "pokelike_b", "red_overworld", "red_battle", "red_bill", "red_pallet"])
def test_cuda_replays_reference_wrapper_recording(cuda_lib, roms, name):
    import torch

    gold = np.load(GOLDEN / f"ref_wrapper_{name}.npz")
    h = _capi.Handle(cuda_lib, 1, roms(str(gold["rom_name"])), 0)
    replay_wrapper_golden(h, gold, to_dev=lambda a: torch.from_numpy(a).cuda(), to_host=lambda t: t.cpu().numpy())


def test_cuda_renderer_matches_pyboy_framebuffers(cuda_lib, roms):
    kat = np.load(GOLDEN / "ppu_kat.npz")
    h = _capi.Handle(cuda_lib, 1, roms("pokelike"), 0)
    check_ppu_kat(h, kat)


def test_cuda_replays_reference_wrapper_on_all_264_states(cuda_lib, roms):
    """Every save-state the reference ships, one env each, in ONE batch (mixed overworld / battle / menu states side by side
    in the same warps): reward, done, observation and final emulator state equal to what the unmodified reference wrapper
    produced."""
    import torch

    gold = load_wrapper_sweep()
    h = _capi.Handle(cuda_lib, len(gold["names"]), roms("pokelike"), 0)
    replay_wrapper_sweep(h, gold, to_dev=lambda a: torch.from_numpy(a).cuda(), to_host=lambda t: t.cpu().numpy())
