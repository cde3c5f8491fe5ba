"""The event-flag table and gbenv_event_flags' oracle form (tests/oracle_ext/oracle_events.c) against info.event_bits over
random WRAM, the info dicts built from event bits against build_info and the reference's recorded dicts, and
event_counts_to_means against per-env dicts.  No GPU."""
import ctypes as C
import json
import re

import numpy as np
import pytest

from helpers import GOLDEN, info_fingerprint
from pokegym_b200 import _capi
from pokegym_b200 import info as I

ROOT = GOLDEN.parent.parent
EW = _capi.EVENT_WORDS
RECORDINGS = ["pokelike_a", "pokelike_b", "red_overworld", "red_battle", "red_bill", "red_pallet"]


def table_entries():
    return [(a, b, w) for g in I.event_table().values() for _, a, b, w in g]


def randomise_wram(h, n, seed):
    """Random bytes in 0xD700-0xD8FF (every event flag's page) of each env; returns the bytes written, [n, 512]."""
    rng = np.random.default_rng(seed)
    data = rng.integers(0, 256, (n, 0x200), dtype=np.uint8)
    for e in range(n):
        h.write_mem(e, 0xD700, data[e])
    return data


def want_bits(h, ids):
    """info.event_bits over the oracle's bus reads, one row per id."""
    out = []
    for e in ids:
        wram = h.read_mem(int(e), 0xD700, 0x200)
        out.append(I.event_bits(lambda a: int(wram[a - 0xD700])))
    return np.stack(out)


def pack(bits):
    """[n, 130] bits -> [n, 5] uint32 words as gbenv_event_flags lays them out."""
    words = np.zeros((len(bits), EW), np.uint32)
    for k in range(_capi.EVENT_FLAGS):
        words[:, k >> 5] |= bits[:, k].astype(np.uint32) << np.uint32(k & 31)
    return words


def replay_info_steps(handle, gold, to_dev=lambda a: a, to_host=lambda a: a):
    """Replays a ref_wrapper_*.npz recording on a 1-env handle and yields (step, info row, recorded fingerprint) at each step
    where the reference emitted an info dict."""
    handle.set_initial_template(handle.add_state_template(gold["start_state"].tobytes()))
    obs = to_dev(np.zeros((1, _capi.OBS_BYTES), np.uint8))
    rew, done = to_dev(np.zeros(1)), to_dev(np.zeros(1, np.uint8))
    row = to_dev(np.zeros((1, _capi.INFO_SCALARS)))
    mes = int(gold["max_episode_steps"])
    reset_at = {int(x) for x in gold["reset_at"]}
    infos = {int(i): json.loads(str(t)) for i, t in zip(gold["info_steps"], gold["info_json"])}
    handle.reset(obs, max_episode_steps=mes)
    for i, a in enumerate(gold["actions"]):
        if i in reset_at:
            handle.reset(obs, max_episode_steps=mes)
        handle.step(to_dev(np.array([a], np.uint8)), obs, rew, done)
        if i in infos:
            handle.get_info(row)
            yield i, to_host(row)[0], infos[i]


def test_event_bits_inc_is_the_event_table():
    text = (ROOT / "pokegym_b200" / "csrc" / "event_bits.inc").read_text()
    body = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("//"))
    entries = [(int(a, 16), int(b), int(w)) for a, b, w in re.findall(r"EV\((0x[0-9A-Fa-f]+),\s*(\d+),\s*(-?\d+)\)", body)]
    assert len(entries) == _capi.EVENT_FLAGS == 130
    assert entries == table_entries()
    assert EW * 32 >= _capi.EVENT_FLAGS > (EW - 1) * 32


def test_event_table_does_not_contain_d778():
    """A non-first reset writes one byte of RAM, D778 bit 4 (k_wrap_reset_pre): with no flag there, a reset leaves every
    event flag as the episode's last step left it, which VecEnvironment.episode_infos relies on after auto_reset."""
    assert all(a != 0xD778 for a, _, _ in table_entries())


@pytest.mark.parametrize("rom_name", ["pokelike", "conformance"])
def test_oracle_event_flags_match_event_bits(oracle_lib, roms, rom_name):
    n = 9
    h = _capi.Handle(oracle_lib, n, roms(rom_name))
    h.tick(3, True)
    randomise_wram(h, n, seed=len(rom_name))
    rng = np.random.default_rng(3)
    everything = want_bits(h, range(n))
    assert everything.any() and not everything.all()
    # NULL ids: envs 0..n-1, also a prefix of them
    for m in (n, 4):
        out = np.zeros((m, EW), np.uint32)
        h.event_flags(out)
        assert np.array_equal(out, pack(everything[:m]))
        assert np.array_equal(I.unpack_event_words(out), everything[:m])
    # any order, duplicates
    ids = np.concatenate([rng.permutation(n), rng.integers(0, n, 7)]).astype(np.int32)
    out = np.zeros((len(ids), EW), np.uint32)
    h.event_flags(out, ids)
    assert np.array_equal(I.unpack_event_words(out), everything[ids])
    assert not (out[:, EW - 1] >> np.uint32(_capi.EVENT_FLAGS - 32 * (EW - 1))).any()  # bits 130..159 are 0
    # out-of-range ids: their rows stay as they were
    ids = np.array([2, -1, n, 5, 1 << 30], np.int32)
    out = np.full((len(ids), EW), 0xA5A5A5A5, np.uint32)
    h.event_flags(out, ids)
    assert (out[[1, 2, 4]] == 0xA5A5A5A5).all()
    assert np.array_equal(out[[0, 3]], pack(everything[[2, 5]]))


def test_oracle_event_flags_error_codes(oracle_lib, roms):
    n = 4
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    lib, out = oracle_lib, np.zeros((n + 1, EW), np.uint32)
    ids = np.zeros(2, np.int32)
    p_out, p_ids = C.c_void_p(out.ctypes.data), C.c_void_p(ids.ctypes.data)
    assert lib.event_flags(None, p_ids, 2, p_out, None) == -1  # GBENV_E_ARG
    assert lib.event_flags(h._h, p_ids, 2, None, None) == -1
    assert lib.event_flags(h._h, p_ids, -1, p_out, None) == -1
    assert lib.event_flags(h._h, None, n + 1, p_out, None) == -1
    assert lib.event_flags(h._h, None, n, p_out, None) == 0
    out[:] = 7
    assert lib.event_flags(h._h, p_ids, 0, p_out, None) == 0  # n == 0: nothing written
    assert lib.event_flags(h._h, None, 0, None, None) == 0
    assert (out == 7).all()
    with pytest.raises(ValueError):  # the binding checks the buffer size before the call
        h.event_flags(np.zeros((1, EW), np.uint32), np.zeros(2, np.int32))
    with pytest.raises(_capi.GbEnvError, match="event_flags"):
        h.event_flags(np.zeros((n + 1, EW), np.uint32))


@pytest.mark.parametrize("name", RECORDINGS)
def test_info_from_event_flags_matches_build_info_and_reference(oracle_lib, roms, name):
    """At every step where the reference emitted an info dict: the dict built from oracle_event_flags equals build_info's
    from bus reads, and both have the reference's fingerprint."""
    gold = np.load(GOLDEN / f"ref_wrapper_{name}.npz")
    h = _capi.Handle(oracle_lib, 1, roms(str(gold["rom_name"])))
    seen = 0
    for i, row, want in replay_info_steps(h, gold):
        wram = h.read_mem(0, 0xD700, 0x200)
        read_byte = lambda a: int(wram[a - 0xD700])  # noqa: E731
        flags = np.zeros((1, EW), np.uint32)
        h.event_flags(flags)
        bits = I.unpack_event_words(flags)[0]
        assert np.array_equal(bits, I.event_bits(read_byte)), i
        cm = h.counts_map(0)
        mine = I.build_info_from_events(row, bits, counts_map=cm)
        assert mine == I.build_info(row, read_byte, counts_map=cm), i
        assert info_fingerprint(mine) == want, i
        seen += 1
    assert seen == len(gold["info_steps"])


def test_event_counts_to_means_is_the_mean_of_per_env_dicts(oracle_lib, roms):
    n = 11
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    randomise_wram(h, n, seed=5)
    bits = want_bits(h, range(n))
    mask = np.array([1, 0, 1, 1, 0, 1, 1, 1, 0, 1, 1], bool)
    row = np.zeros(_capi.INFO_SCALARS)
    dicts = [I.build_info_from_events(row, bits[e]) for e in np.nonzero(mask)[0]]
    means = I.event_counts_to_means(bits[mask].sum(0, dtype=np.int64), int(mask.sum()))
    assert set(means) == {k for k in dicts[0] if k.startswith("detailed_rewards_") or k.endswith("_aggregate") or k == "gym_events"}

    def walk(m, ds, path):
        if isinstance(m, dict):
            assert list(m) == list(ds[0]), path
            for k in m:
                walk(m[k], [d[k] for d in ds], path + (k,))
        else:
            assert np.isclose(m, np.mean(ds), rtol=1e-12, atol=0), (path, m, np.mean(ds))

    walk(means, [{k: d[k] for k in means} for d in dicts], ())
    assert any(v != 0 for v in means["dojo_events_aggregate"].values())
    zero = I.event_counts_to_means(np.zeros(130, np.int64), 0)  # no env: zeros, not a division by zero
    assert all(v == 0.0 for v in zero["dojo_events_aggregate"].values())
    with pytest.raises(ValueError):
        I.event_counts_to_means(np.zeros(129), 1)
