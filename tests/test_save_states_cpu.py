"""The v9 section table of csrc/gb_image.h (STATE_LAYOUT), which both the host serialiser (image_to_blob) and the device one
(k_save_states) read, against pokegym_b200.state_file: its sections tile the file along the field boundaries of
state_file.field_offsets, and serialising the committed fixtures through it gives back state_file.serialize_state's bytes.
Also gbenv_save_states' argument rules on the CPU oracle."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from helpers import GOLDEN, ppu_kat_blob, ppu_kat_expected_screen
from pokegym_b200 import _capi
from pokegym_b200.state_file import field_offsets, parse_state, serialize_state

SRC = GOLDEN.parent / "hostsim" / "state_table.cpp"
S = _capi.STATE_BYTES
KINDS = ("const", "field", "bytes", "lp", "fb")


@pytest.fixture(scope="module")
def table(tmp_path_factory):
    out = tmp_path_factory.mktemp("state_table") / "libstate_table.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(out), str(SRC)], check=True)
    dll = C.CDLL(str(out))
    dll.st_sections.argtypes = [C.c_void_p]
    dll.st_section_of.argtypes = [C.c_uint32]
    dll.st_roundtrip.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p]
    return dll


def _sections(dll):
    buf = np.zeros((64, 6), np.uint32)
    k = dll.st_sections(buf.ctypes.data)
    return [dict(off=int(r[0]), len=int(r[1]), src=int(r[2]), kind=KINDS[r[3]], shift=int(r[4]), mask=int(r[5])) for r in buf[:k]]


def _roundtrip(dll, blob: bytes) -> bytes:
    out = np.zeros(S, np.uint8)
    assert dll.st_roundtrip(blob, len(blob), out.ctypes.data) == 0
    return out.tobytes()


def test_sections_tile_the_file_along_state_file_fields(table):
    secs = _sections(table)
    off = 0
    for s in secs:
        assert s["off"] == off and s["len"] > 0
        off += s["len"]
    assert off == S
    starts = {s["off"] for s in secs}
    for name, (o, ln) in field_offsets(9).items():
        assert o in starts, f"field {name} starts inside a section"
        assert o + ln in starts | {S}, f"field {name} ends inside a section"
    by_off = {s["off"]: s for s in secs}
    f = field_offsets(9)
    assert by_off[f["vram"][0]]["kind"] == "bytes" and by_off[f["vram"][0]]["len"] == 0x2000 and f["vram"][0] == 23
    assert by_off[f["wram"][0]]["kind"] == "bytes" and f["wram"][0] == 101_285
    assert by_off[f["screen"][0]]["kind"] == "fb" and by_off[f["screen"][0]]["len"] == f["screen"][1]
    assert by_off[f["scanline_params"][0]]["kind"] == "lp" and by_off[f["scanline_params"][0]]["len"] == f["scanline_params"][1]
    assert by_off[f["cart_ram"][0]]["len"] == 0x8000 and by_off[0]["kind"] == "const" and by_off[0]["src"] == 9


def test_section_lookup(table):
    secs = _sections(table)
    for i, s in enumerate(secs):
        for o in {s["off"], s["off"] + s["len"] // 2, s["off"] + s["len"] - 1}:
            assert table.st_section_of(o) == i, o


def test_mixed_states_serialise_like_state_file(table):
    states = np.load(GOLDEN / "red_states_mixed.npz")["states"]
    for i, row in enumerate(states):
        blob = serialize_state(parse_state(row.tobytes()))
        assert blob == row.tobytes()
        got = _roundtrip(table, blob)
        if got != blob:
            bad = np.nonzero(np.frombuffer(got, np.uint8) != row)[0]
            raise AssertionError(f"state {i}: {bad.size} bytes differ, first at offset {bad[0]}")


def test_ppu_kat_states_serialise_like_state_file(table):
    kat = np.load(GOLDEN / "ppu_kat.npz")
    base = np.load(GOLDEN / "red_states_mixed.npz")["states"][0].tobytes()
    for i in range(len(kat["names"])):
        st = parse_state(ppu_kat_blob(base, kat, i))
        st.raw["screen"] = np.frombuffer(ppu_kat_expected_screen(kat, i), np.uint8)
        blob = serialize_state(st)
        assert _roundtrip(table, blob) == blob, kat["names"][i]


def test_oracle_save_states_rows_and_arguments(oracle_lib, roms):
    n = 37
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    h.tick(3, True)
    want = np.stack([np.frombuffer(h.save_state(e), np.uint8) for e in range(n)])
    out = np.zeros((n, S), np.uint8)
    h.save_states(out)
    assert np.array_equal(out, want)
    ids = np.array([5, -1, n, 0, 5], np.int32)
    rows = np.full((5, S), 0x5A, np.uint8)
    h.save_states(rows, ids)
    assert np.array_equal(rows[[0, 3, 4]], want[[5, 0, 5]]) and (rows[[1, 2]] == 0x5A).all()
    h.save_states(np.zeros((0, S), np.uint8))
    with pytest.raises(ValueError):
        h.save_states(np.zeros((n, S - 1), np.uint8))
    with pytest.raises(_capi.GbEnvError):
        h.save_states(np.zeros((n + 1, S), np.uint8))
