"""The v9 parser k_load_states runs (state_image_word and state_row_valid in csrc/gb_image.h, driven by the same section
table as the serialiser) against the hand-written host parser blob_to_image, which gbenv_add_state_template uses: the same
image for the committed fixtures and for rows with random RAM, register and field bytes, and the same accept / reject
decision on corrupted rows.  Also gbenv_load_states' contract on the CPU oracle."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from helpers import GOLDEN, ppu_kat_blob, ppu_kat_expected_screen
from pokegym_b200 import _capi
from pokegym_b200.state_file import field_offsets, parse_state, serialize_state

SRC = GOLDEN.parent / "hostsim" / "load_table.cpp"
S = _capi.STATE_BYTES
E_ARG, E_STATE = -1, -2
F = field_offsets(9)


@pytest.fixture(scope="module")
def table(tmp_path_factory):
    out = tmp_path_factory.mktemp("load_table") / "libload_table.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(out), str(SRC)], check=True)
    dll = C.CDLL(str(out))
    dll.st_image_from_row.argtypes = [C.c_void_p, C.c_void_p]
    dll.st_blob_to_image.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
    dll.st_row_valid.argtypes = [C.c_void_p]
    return dll


def _row(blob) -> np.ndarray:
    return np.ascontiguousarray(np.frombuffer(bytes(blob), np.uint8))


def _images(dll, blob):
    row = _row(blob)
    n = dll.st_img_words()
    ref, got = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
    rc = dll.st_blob_to_image(row.ctypes.data, row.size, ref.ctypes.data)
    dll.st_image_from_row(row.ctypes.data, got.ctypes.data)
    return rc, ref, got


def _same_image(dll, blob, what):
    rc, ref, got = _images(dll, blob)
    assert rc == 0, what
    bad = np.nonzero(ref != got)[0]
    assert bad.size == 0, f"{what}: {bad.size} image words differ, first {bad[0]}: {ref[bad[0]]:#x} vs {got[bad[0]]:#x}"
    assert table_valid(dll, blob), what


def table_valid(dll, blob) -> bool:
    row = _row(blob)
    return bool(dll.st_row_valid(row.ctypes.data))


def _mixed():
    return np.load(GOLDEN / "red_states_mixed.npz")["states"]


def test_mixed_states_parse_like_blob_to_image(table):
    for i, row in enumerate(_mixed()):
        _same_image(table, row.tobytes(), f"state {i}")


def test_ppu_kat_states_parse_like_blob_to_image(table):
    kat = np.load(GOLDEN / "ppu_kat.npz")
    base = _mixed()[0].tobytes()
    for i in range(len(kat["names"])):
        st = parse_state(ppu_kat_blob(base, kat, i))
        st.raw["screen"] = np.frombuffer(ppu_kat_expected_screen(kat, i), np.uint8)
        _same_image(table, serialize_state(st), kat["names"][i])


# every field but the version byte, the cgb byte and the high halves of the two LCD clocks takes any byte value; the screen
# takes any of the four shade words
CLOCK_HIGH = [F["lcd_clock"][0] + 2 + 4 + k for k in range(4)] + [F["lcd_clock"][0] + 2 + 8 + 4 + k for k in range(4)]
SHADES = np.array([0xFFFFFF01, 0x99999900, 0x55555500, 0x00000000], np.uint32)


def _randomised(rng, base):
    row = base.copy()
    for name, (o, ln) in F.items():
        if name != "screen":
            row[o : o + ln] = rng.integers(0, 256, ln, dtype=np.uint8)
    o, ln = F["screen"]
    row[o : o + ln] = SHADES[rng.integers(0, 4, ln // 4)].view(np.uint8)
    row[0], row[4] = 9, 0
    row[CLOCK_HIGH] = 0
    return row


def test_random_ram_register_and_field_bytes(table):
    rng = np.random.default_rng(9)
    base = _mixed()
    for t in range(24):
        _same_image(table, _randomised(rng, base[t % len(base)]).tobytes(), f"random {t}")


def _corruptions(row):
    """(name, corrupted copy) for every byte blob_to_image checks, plus screen words set to a fifth value"""
    so = F["screen"][0]
    for name, o, v in [("version", 0, 7), ("version", 0, 0), ("cgb", 4, 1), ("cgb", 4, 0x80)] + [(f"clock high {o}", o, 1) for o in CLOCK_HIGH]:
        bad = row.copy()
        bad[o] = v
        yield name, bad
    for k, w in [(0, 0xFFFFFF00), (1, 0x99999901), (23039, 0x12345678), (11520, 0x00000001), (7, 0x55555501)]:
        bad = row.copy()
        bad[so + 4 * k : so + 4 * k + 4] = np.array([w], np.uint32).view(np.uint8)
        yield f"screen word {k}", bad


def test_validity_predicate_agrees_with_blob_to_image(table):
    rng = np.random.default_rng(3)
    rows = list(_mixed()[:6]) + [_randomised(rng, _mixed()[7])]
    for row in rows:
        rc, _, _ = _images(table, row.tobytes())
        assert rc == 0 and table_valid(table, row.tobytes())
        for name, bad in _corruptions(row):
            rc, _, _ = _images(table, bad.tobytes())
            assert rc == E_STATE, name
            assert not table_valid(table, bad.tobytes()), name
    # the second copies of cgb and double_speed after the LCD registers are not checked (blob_to_image ignores them)
    row = _mixed()[0].copy()
    row[F["lcd_clock"][0]] = 1
    assert _images(table, row.tobytes())[0] == 0 and table_valid(table, row.tobytes())


def _oracle(oracle_lib, roms, n):
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    h.tick(3, True)
    return h


def _rows(h, n):
    out = np.zeros((n, S), np.uint8)
    h.save_states(out)
    return out


def test_oracle_load_states_contract(oracle_lib, roms):
    n = 12
    src = _oracle(oracle_lib, roms, n)
    states = _mixed()
    for e in range(n):
        src.load_template(src.add_state_template(states[e].tobytes()), [e])
    want = _rows(src, n)
    bad = want[3].copy()
    bad[4] = 1  # cgb
    dst = _oracle(oracle_lib, roms, n)
    before = _rows(dst, n)
    # 5 <- row 0 then row 1 (last valid wins), 6 <- valid row 2 then a corrupt row (the earlier one stays), 7 <- only corrupt,
    # -1 and n skipped
    ids = np.array([5, 5, 6, 6, 7, -1, n, 0], np.int32)
    blobs = np.stack([want[0], want[1], want[2], bad, bad, want[4], want[5], want[8]])
    status = np.full(len(ids), 99, np.int32)
    dst.load_states(blobs, ids, status)
    assert status.tolist() == [0, 0, 0, E_STATE, E_STATE, E_ARG, E_ARG, 0]
    got = _rows(dst, n)
    ref = _oracle(oracle_lib, roms, n)
    for e, k in ((5, 1), (6, 2), (0, 8)):
        ref.load_template(ref.add_state_template(want[k].tobytes()), [e])
    assert np.array_equal(got, _rows(ref, n))
    assert np.array_equal(got[7], before[7]) and np.array_equal(got[[1, 2, 3, 4, 8, 9, 10, 11]], before[[1, 2, 3, 4, 8, 9, 10, 11]])
    # NULL ids: envs 0..k-1; status optional
    dst.load_states(want[:4])
    for e in range(4):
        ref.load_template(ref.add_state_template(want[e].tobytes()), [e])
    assert np.array_equal(_rows(dst, n), _rows(ref, n))
    # argument rules
    lib, hp = oracle_lib, dst._h
    p = blobs.ctypes.data
    assert lib.load_states(None, None, 1, C.c_void_p(p), None, None) == E_ARG
    assert lib.load_states(hp, None, 1, None, None, None) == E_ARG
    assert lib.load_states(hp, None, -1, C.c_void_p(p), None, None) == E_ARG
    assert lib.load_states(hp, None, n + 1, C.c_void_p(p), None, None) == E_ARG
    assert lib.load_states(hp, C.c_void_p(ids.ctypes.data + 2), 1, C.c_void_p(p), None, None) == E_ARG
    assert lib.load_states(hp, None, 1, C.c_void_p(p), C.c_void_p(status.ctypes.data + 1), None) == E_ARG
    assert lib.load_states(hp, None, 0, None, None, None) == 0
    with pytest.raises(ValueError):
        dst.load_states(blobs[:, :-1].copy(), ids)
    with pytest.raises(ValueError):
        dst.load_states(blobs, ids[:3])
    with pytest.raises(ValueError):
        dst.load_states(blobs, ids, np.zeros(len(ids), np.int64))
