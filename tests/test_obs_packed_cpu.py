"""Packed observations on the CPU oracle: every reference observation fits the packed layout, oracle_unpack_obs gives it back
byte for byte, and the oracle's packed rows equal a packer written here from the layout text of include/gbenv.h; the
argument checks of the three calls and of the Python binding."""
import numpy as np
import pytest

from pokegym_b200 import _capi

GREY = np.array([0xFF, 0x99, 0x55, 0x00], np.uint8)
E_ARG = -1  # GBENV_E_ARG
PB, OB = _capi.OBS_PACKED_BYTES, _capi.OBS_BYTES
SENTINEL = 0xA5


def aligned(shape, dtype=np.uint8, offset=0):
    """A zeroed C-contiguous array whose data starts `offset` bytes past a 64-byte boundary."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    raw = np.zeros(nbytes + 64 + offset, np.uint8)
    start = (-raw.ctypes.data) % 64 + offset
    return raw[start:start + nbytes].view(dtype).reshape(shape)


def np_pack(obs):
    """uint8 [n, 72, 80, 4] reference observations -> uint32 [n, 576], from the header's words: row i is words 8i .. 8i+7;
    word 8i+k (k < 5) holds the shade of pixel j = 16k + t at bit 2t, word 8i+5+m the visited bit of pixel 32m + b at bit b."""
    lut = np.full(256, 255, np.uint64)
    lut[GREY] = np.arange(4)
    shade = lut[obs[..., 0]]  # [n, 72, 80]
    vis = (obs[..., 3] != 0).astype(np.uint64)
    words = np.zeros(obs.shape[:2] + (8,), np.uint64)
    for k in range(5):
        words[..., k] = (shade[..., 16 * k:16 * k + 16] << (2 * np.arange(16, dtype=np.uint64))).sum(-1)
    for m in range(3):
        cols = np.arange(32 * m, min(32 * m + 32, 80))
        words[..., 5 + m] = (vis[..., cols] << (cols - 32 * m).astype(np.uint64)).sum(-1)
    return words.astype(np.uint32).reshape(len(obs), -1)


def check_reference_obs(obs):
    """Channels 0-2 equal and one of the four greys, channel 3 0 or 255: what makes 3 bits per pixel lossless."""
    o = obs.reshape(-1, 72, 80, 4)
    assert (o[..., 0] == o[..., 1]).all() and (o[..., 0] == o[..., 2]).all()
    assert np.isin(o[..., 0], GREY).all()
    assert np.isin(o[..., 3], [0, 255]).all()


def check_rows(h, obs, packed, rows):
    if len(rows) == 0:
        return
    check_reference_obs(obs[rows])
    assert np.array_equal(packed[rows].view(np.uint32), np_pack(obs[rows].reshape(-1, 72, 80, 4)))
    out = aligned((len(rows), OB))
    h.unpack_obs(packed[rows], out)
    assert np.array_equal(out, obs[rows])


def twin_run(oracle_lib, rom, n, steps, blobs=None, mes=6, seed=0):
    """Handle `ref` steps / resets with the reference calls, `pk` with the packed ones, same actions, skips and resets."""
    ref, pk = _capi.Handle(oracle_lib, n, rom), _capi.Handle(oracle_lib, n, rom)
    for h in (ref, pk):
        if blobs is None:
            h.tick(30, True)
        else:
            for k, blob in enumerate(blobs):
                h.set_initial_template(h.add_state_template(blob), np.arange(k, n, len(blobs), dtype=np.int32))
    obs, packed = aligned((n, OB)), aligned((n, PB))
    ra, rb, da, db = np.zeros(n), np.zeros(n), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    ref.reset(obs, max_episode_steps=mes)
    pk.reset_packed(packed, max_episode_steps=mes)
    every = np.arange(n)
    check_rows(pk, obs, packed, every)
    rng = np.random.default_rng(seed)
    visited = 0
    for s in range(steps):
        act = rng.integers(0, 8, n).astype(np.uint8)
        skip = (rng.random(n) < 0.3).astype(np.uint8) if s % 2 else None
        if skip is not None:  # the rows of envs that sit out must come back untouched
            obs[skip.astype(bool)] = SENTINEL
            packed[skip.astype(bool)] = SENTINEL
        ref.step_masked(act, skip, obs, ra, da)
        pk.step_packed(act, skip, packed, rb, db)
        assert np.array_equal(ra, rb) and np.array_equal(da, db), f"step {s}"
        stepped = every if skip is None else np.nonzero(skip == 0)[0]
        check_rows(pk, obs, packed, stepped)
        if skip is not None:
            assert (packed[skip.astype(bool)] == SENTINEL).all()
        visited += int((obs.reshape(n, 72, 80, 4)[stepped, ..., 3] != 0).sum())
        if da.any():
            ref.reset(obs, mask=da, max_episode_steps=mes)
            pk.reset_packed(packed, mask_dev=da, max_episode_steps=mes)
            check_rows(pk, obs, packed, np.nonzero(da)[0])
    assert visited > 0  # the visited channel was exercised
    for e in range(n):
        assert ref.save_state(e) == pk.save_state(e), e
    return ref, pk


@pytest.mark.parametrize("rom_name", ["pokelike", "lcd_probe"])
def test_oracle_packed_twin_run(oracle_lib, roms, rom_name):
    twin_run(oracle_lib, roms(rom_name), n=6, steps=14, mes=5, seed=len(rom_name))


def test_oracle_packed_twin_run_mixed_reference_states(oracle_lib, roms):
    """The 40 reference save-states (overworld, battles, menus, many maps): visited windows at map edges."""
    from helpers import GOLDEN

    blobs = [b.tobytes() for b in np.load(GOLDEN / "red_states_mixed.npz")["states"]]
    twin_run(oracle_lib, roms("pokelike"), n=len(blobs), steps=8, blobs=blobs, mes=3, seed=40)


def test_np_pack_follows_the_layout_on_single_pixels():
    obs = np.zeros((1, 72, 80, 4), np.uint8)
    obs[..., :3] = 0xFF  # shade 0 everywhere
    obs[0, 5, 37, :3] = 0x55  # shade 2 at (5, 37): word 8*5 + 2, bit 2 * 5
    obs[0, 71, 79, 3] = 255  # visited (71, 79): word 8*71 + 7, bit 15
    w = np_pack(obs)[0]
    assert w[8 * 5 + 2] == 2 << 10 and w[8 * 71 + 7] == 1 << 15
    assert np.count_nonzero(w) == 2


def test_oracle_packed_argument_errors(oracle_lib, roms):
    n = 4
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    lib, hh, vp = h.lib, h._h, _capi._ptr
    act, rew, done = np.zeros(n, np.uint8), np.zeros(n), np.zeros(n, np.uint8)
    packed, out = aligned((n, PB)), aligned((n, OB))
    bad_p, bad_o = aligned((n, PB), offset=4), aligned((n, OB), offset=8)
    assert lib.step_packed(None, vp(act), None, vp(packed), vp(rew), vp(done), None) == E_ARG
    for args in ((None, None, vp(packed), vp(rew), vp(done)), (vp(act), None, None, vp(rew), vp(done)), (vp(act), None, vp(packed), None, vp(done)),
                 (vp(act), None, vp(packed), vp(rew), None), (vp(act), None, vp(bad_p), vp(rew), vp(done))):
        assert lib.step_packed(hh, *args, None) == E_ARG
    assert lib.reset_packed(hh, None, 100, 4.0, None, None) == E_ARG
    assert lib.reset_packed(hh, None, 100, 4.0, vp(bad_p), None) == E_ARG
    assert lib.reset_packed(None, None, 100, 4.0, vp(packed), None) == E_ARG
    assert lib.unpack_obs(hh, vp(packed), -1, vp(out), None) == E_ARG
    assert lib.unpack_obs(hh, None, 1, vp(out), None) == E_ARG
    assert lib.unpack_obs(hh, vp(packed), 1, None, None) == E_ARG
    assert lib.unpack_obs(hh, vp(bad_p), 1, vp(out), None) == E_ARG
    assert lib.unpack_obs(hh, vp(packed), 1, vp(bad_o), None) == E_ARG
    assert lib.unpack_obs(None, vp(packed), 1, vp(out), None) == E_ARG
    out[:] = SENTINEL
    assert lib.unpack_obs(hh, None, 0, None, None) == 0  # n == 0: a no-op
    assert lib.unpack_obs(hh, vp(packed), 0, vp(out), None) == 0
    assert (out == SENTINEL).all()
    # the binding refuses a buffer of the wrong type, size, layout or alignment before any pointer crosses the ABI
    for bad in (bad_p, packed[:n - 1], packed.view(np.uint32), aligned((PB, n)).T):
        with pytest.raises(ValueError):
            h.step_packed(act, None, bad, rew, done)
        with pytest.raises(ValueError):
            h.reset_packed(bad)
    with pytest.raises(ValueError):
        h.unpack_obs(packed, out[:n - 1])
    with pytest.raises(ValueError):
        h.unpack_obs(packed[:, :100], out)
    with pytest.raises(ValueError):
        h.unpack_obs(packed, bad_o)
    with pytest.raises(TypeError):
        h.unpack_obs(bytes(PB), out[:1])
