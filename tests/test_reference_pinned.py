"""Pin the state codec and the oracle to what the reference itself holds: its 264 PyBoy v9 save-states, stored unmodified
in tests/golden/ref_wrapper_sweep.npz (helpers.load_wrapper_sweep) and named by their path in the reference tree."""
from helpers import load_wrapper_sweep
from pokegym_b200 import _capi
from pokegym_b200.state_file import diff_states, parse_state, serialize_state


def _fixtures():
    gold = load_wrapper_sweep()
    return [(str(name), state.tobytes()) for name, state in zip(gold["names"], gold["states"])]


def test_state_codec_round_trips_every_fixture():
    fixtures = _fixtures()
    assert len(fixtures) == 264
    for name, blob in fixtures:
        assert serialize_state(parse_state(blob)) == blob, name


def test_oracle_load_save_and_renderer_on_all_v9_fixtures(oracle_lib, roms):
    """gb_load_state/gb_save_state are byte-exact (except STAT's read-only low bits, a PyBoy load quirk) and the
    scanline renderer reproduces, bit for bit, the framebuffer PyBoy stored in each of the 264 save-states."""
    h = _capi.Handle(oracle_lib, 1, roms("pokelike"))
    fixtures = _fixtures()
    assert len(fixtures) == 264
    for name, blob in fixtures:
        tid = h.add_state_template(blob)
        h.load_template(tid)
        d = diff_states(blob, h.save_state(0))
        assert d in ([], ["lcd_regs: 1 bytes differ (+4:81!=80)"]), (name, d)
        expected = parse_state(blob).raw["screen"].tobytes()
        h.debug_render_frame(0)
        assert parse_state(h.save_state(0)).raw["screen"].tobytes() == expected, f"{name}: rendered frame differs from PyBoy's"
