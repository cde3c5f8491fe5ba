"""Batched frames on the CPU oracle: oracle_capture_frames / oracle_frames_to_rgb give oracle_screen byte for byte, their
argument checks, and the chronological order of FrameRecorder's ring."""
import numpy as np
import pytest

from pokegym_b200 import _capi

GREY = np.array([0xFF, 0x99, 0x55, 0x00], np.uint8)
E_ARG = -1  # GBENV_E_ARG


def _capture(h, ids=None, n=None):
    n = len(ids) if ids is not None else n
    frames = np.zeros((n, _capi.FRAME_WORDS), np.uint32)
    h.capture_frames(frames, None if ids is None else np.ascontiguousarray(ids, np.int32))
    return frames


def _decode(h, frames, channels):
    out = np.zeros((len(frames), _capi.SCREEN_H, _capi.SCREEN_W, channels), np.uint8)
    h.frames_to_rgb(frames, out, channels)
    return out


def _check_against_screen(h, ids):
    frames = _capture(h, ids)
    rgb, grey = _decode(h, frames, 3), _decode(h, frames, 1)
    for k, e in enumerate(ids):
        want = h.screen(int(e))
        assert np.array_equal(rgb[k], want), (k, e)
        assert np.array_equal(grey[k, ..., 0], want[..., 0]), (k, e)
        # the packed format itself: pixel (x, y) is the 2-bit shade at bit 2 * (x & 15) of word y * 10 + x / 16
        y, x = 77, 133
        shade = (int(frames[k, y * 10 + x // 16]) >> (2 * (x & 15))) & 3
        assert GREY[shade] == want[y, x, 0]
    return frames


@pytest.mark.parametrize("rom_name", ["pokelike", "lcd_probe", "conformance"])
def test_oracle_capture_and_decode_equal_screen(oracle_lib, roms, rom_name):
    n = 9
    h = _capi.Handle(oracle_lib, n, roms(rom_name))
    rng = np.random.default_rng(3)
    ids = np.array([7, 2, 2, 8, 0, 5, 7, 1], np.int32)  # any order, duplicates
    h.tick(2, True)
    _check_against_screen(h, ids)
    obs, rew, done = np.zeros((n, _capi.OBS_BYTES), np.uint8), np.zeros(n), np.zeros(n, np.uint8)
    h.reset(obs)
    distinct = set()
    for s in range(6):
        h.step(rng.integers(0, 8, n).astype(np.uint8), obs, rew, done)
        frames = _check_against_screen(h, rng.permutation(n).astype(np.int32))
        distinct.update(f.tobytes() for f in frames)
    assert np.array_equal(_capture(h, n=n), _capture(h, np.arange(n)))  # NULL ids: envs 0..n-1
    if rom_name != "conformance":  # that ROM exercises the CPU and leaves the screen blank
        assert len(distinct) > 1  # the frames compared are not all the same picture
    lcd_off_on(h, n, lambda: _check_against_screen(h, ids))


def lcd_off_on(h, n, check):
    """The LCD of the odd envs switched off (LCDC bit 7) for two frames, then back to its LCDC for two; `check` after each."""
    lcdc = [int(h.read_mem(e, 0xFF40)[0]) for e in range(n)]
    for e in range(1, n, 2):
        h.write_mem(e, 0xFF40, [lcdc[e] & 0x7F])
    h.tick(2, True)
    check()
    for e in range(1, n, 2):
        h.write_mem(e, 0xFF40, [lcdc[e]])
    h.tick(2, True)
    check()


def test_oracle_frame_argument_errors_and_untouched_rows(oracle_lib, roms):
    n = 4
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    h.tick(2, True)
    lib, hh = h.lib, h._h
    frames = np.full((3, _capi.FRAME_WORDS), 0xDEADBEEF, np.uint32)
    ids = np.array([1, -1, 4], np.int32)  # only the first is valid
    h.capture_frames(frames, ids)
    assert np.array_equal(frames[0], _capture(h, [1])[0])
    assert (frames[1:] == 0xDEADBEEF).all()
    out = np.zeros((1, 144, 160, 3), np.uint8)
    vp = _capi._ptr
    assert lib.capture_frames(hh, None, n + 1, vp(np.zeros((n + 1, _capi.FRAME_WORDS), np.uint32)), None) == E_ARG  # NULL ids, n > n_envs
    assert lib.capture_frames(hh, None, -1, vp(frames), None) == E_ARG
    assert lib.capture_frames(hh, None, 1, None, None) == E_ARG
    assert lib.capture_frames(None, None, 1, vp(frames), None) == E_ARG
    assert lib.capture_frames(hh, None, 0, None, None) == 0  # n == 0: a no-op
    for ch in (0, 2, 4):
        assert lib.frames_to_rgb(hh, vp(frames), 1, ch, vp(out), None) == E_ARG
    assert lib.frames_to_rgb(hh, vp(frames), -1, 3, vp(out), None) == E_ARG
    assert lib.frames_to_rgb(hh, None, 1, 3, vp(out), None) == E_ARG
    assert lib.frames_to_rgb(hh, vp(frames), 1, 3, None, None) == E_ARG
    assert lib.frames_to_rgb(hh, None, 0, 3, None, None) == 0
    with pytest.raises(_capi.GbEnvError):
        h.frames_to_rgb(frames[:1], out, channels=2)
    with pytest.raises(ValueError):  # the binding checks buffer sizes before raw pointers cross the ABI
        h.frames_to_rgb(frames, out)
    with pytest.raises(ValueError):
        h.capture_frames(frames[:2], np.arange(3, dtype=np.int32))


class _Ring:
    """FrameRecorder's bookkeeping without a device: only the fields _segments reads."""

    def __init__(self, capacity, recorded):
        from pokegym_b200.frames import FrameRecorder

        self.r = object.__new__(FrameRecorder)
        self.r.capacity, self.r._recorded = capacity, recorded

    def order(self, start=0, stop=None):
        return [s for a, b in self.r._segments(start, stop) for s in range(a, b)]


@pytest.mark.parametrize("capacity,recorded", [(5, 0), (5, 3), (5, 5), (5, 7), (5, 10), (5, 13), (1, 4)])
def test_recorder_ring_order_is_chronological(capacity, recorded):
    ring = _Ring(capacity, recorded)
    first = max(0, recorded - capacity)  # the oldest step still held
    want = [t % capacity for t in range(first, recorded)]  # step t went to slot t mod capacity
    assert ring.r.count == len(want)
    assert ring.order() == want
    for start, stop in ((1, None), (0, 2), (-2, None), (2, -1), (3, 3)):
        assert ring.order(start, stop) == want[start:stop], (start, stop)
    assert len(ring.r._segments()) <= 2


def test_host_env_ids_are_checked():
    from pokegym_b200.frames import check_channels, host_env_ids

    assert host_env_ids([3, 0, 3], 4).dtype == np.int32
    for bad in ([], [0, 4], [-1], [[0, 1]], [0.5]):
        with pytest.raises(ValueError):
            host_env_ids(bad, 4)
    with pytest.raises(ValueError):
        check_channels(2)
