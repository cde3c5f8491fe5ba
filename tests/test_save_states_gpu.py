"""Batched save-states on the device (gbenv_save_states / k_save_states, and gbenv_save_state, now one launch of the same
kernel): every row is the env's PyBoy v9 file, bit-identical to gbenv_save_state and to the CPU oracle, for any ids, at any
row alignment, across streams; the files load back; the screen field is the packed frame; and saving changes nothing."""
import ctypes as C

import numpy as np
import pytest

from helpers import GOLDEN, SHADE_WORDS
from pokegym_b200 import _capi
from pokegym_b200.state_file import diff_states, field_offsets

pytestmark = pytest.mark.gpu

S = _capi.STATE_BYTES
SENTINEL = 0xA7


def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _mixed(h, n):
    """env i starts from mixed reference state i mod 40"""
    states = np.load(GOLDEN / "red_states_mixed.npz")["states"]
    for k, blob in enumerate(states):
        ids = np.arange(k, n, len(states), dtype=np.int32)
        if ids.size:
            h.load_template(h.add_state_template(blob.tobytes()), ids)


def _gpu_rows(h, n, ids=None, stream=None):
    import torch

    out = torch.full((n, S), SENTINEL, dtype=torch.uint8, device="cuda")
    h.save_states(out, None if ids is None else _dev(np.asarray(ids, np.int32)), stream=stream)
    return out.cpu().numpy()


def _cpu_rows(h, n):
    out = np.zeros((n, S), np.uint8)
    h.save_states(out)
    return out


def _single(h, n):
    return np.stack([np.frombuffer(h.save_state(e), np.uint8) for e in range(n)])


def _first_diff(a, b, where):
    bad = [i for i in range(len(a)) if not np.array_equal(a[i], b[i])]
    if bad:
        raise AssertionError(f"{where}: {len(bad)} rows differ, first env {bad[0]}: {diff_states(a[bad[0]].tobytes(), b[bad[0]].tobytes())[:4]}")


@pytest.mark.parametrize("rom_name,n,mixed", [("pokelike", 1, True), ("pokelike", 31, True), ("pokelike", 33, True),
                                              ("conformance", 33, False), ("pokelike", 4096, True)])
def test_rows_match_single_env_call_and_oracle(cuda_lib, oracle_lib, roms, rom_name, n, mixed):
    rom = roms(rom_name)
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    for h in (gpu, cpu):
        if mixed:
            _mixed(h, n)
        else:
            h.tick(30, True)
    rng = np.random.default_rng(n)
    done = 0
    for steps in (0, 1, 50):
        for _ in range(steps - done):
            act = rng.integers(0, 8, n).astype(np.uint8)
            gpu.run_action(_dev(act))
            cpu.run_action(act)
        done = steps
        rows = _gpu_rows(gpu, n)
        _first_diff(rows, _single(gpu, n), f"{steps} steps: gbenv_save_state")
        _first_diff(rows, _cpu_rows(cpu, n), f"{steps} steps: oracle")
    if mixed:
        assert len({r.tobytes() for r in rows}) >= min(n, 40)  # the envs really differ


def test_id_semantics_and_row_alignment(cuda_lib, roms):
    import torch

    n = 70
    h = _capi.Handle(cuda_lib, n, roms("pokelike"), 0)
    _mixed(h, n)
    rng = np.random.default_rng(5)
    for _ in range(2):
        h.run_action(_dev(rng.integers(0, 8, n).astype(np.uint8)))
    want = _single(h, n)
    assert np.array_equal(_gpu_rows(h, n), want)  # NULL ids, rows at every offset 2i (mod 16) of an aligned base
    for ids in (np.arange(n)[::-1], np.arange(0, n, 3), np.array([7, 7, 0, 69, 7, 1] * 5), np.arange(9, 69)):
        assert np.array_equal(_gpu_rows(h, len(ids), ids), want[ids]), ids[:8]
    assert np.array_equal(_gpu_rows(h, 40), want[:40])  # NULL ids with n < n_envs
    # out-of-range ids keep the sentinel, including the bytes of their rows that share a 16-byte unit with a valid row
    ids = np.array([3, -1, 4, n, n, 5, 1 << 30, 6, -1], np.int32)
    rows = _gpu_rows(h, len(ids), ids)
    ok = ids >= 0
    ok &= ids < n
    assert (rows[~ok] == SENTINEL).all()
    assert np.array_equal(rows[ok], want[ids[ok]])
    # nothing is written past the last row
    buf = torch.full((6, S), SENTINEL, dtype=torch.uint8, device="cuda")
    h.save_states(buf[:5], _dev(np.array([1, 2, 3, 4, 5], np.int32)))
    b = buf.cpu().numpy()
    assert np.array_equal(b[:5], want[1:6]) and (b[5] == SENTINEL).all()
    # n == 0 is a no-op
    h.save_states(torch.empty((0, S), dtype=torch.uint8, device="cuda"))
    h.save_states(torch.empty((0, S), dtype=torch.uint8, device="cuda"), _dev(np.zeros(0, np.int32)))


def test_argument_errors(cuda_lib, roms):
    import torch

    n = 40
    h = _capi.Handle(cuda_lib, n, roms("pokelike"), 0)
    buf = torch.zeros((n + 2) * S + 16, dtype=torch.uint8, device="cuda")
    ids = _dev(np.arange(4, dtype=np.int32))
    p, hp, lib = buf.data_ptr(), h._h, cuda_lib
    E = -1  # GBENV_E_ARG
    assert lib.save_states(None, None, 4, C.c_void_p(p), None) == E  # NULL handle
    assert lib.save_states(hp, None, 4, None, None) == E  # NULL output, n > 0
    for mis in (1, 2, 8):
        assert lib.save_states(hp, None, 4, C.c_void_p(p + mis), None) == E  # output not 16-byte aligned
    assert lib.save_states(hp, None, -1, C.c_void_p(p), None) == E  # n < 0
    assert lib.save_states(hp, None, n + 1, C.c_void_p(p), None) == E  # NULL ids with n > n_envs
    assert lib.save_states(hp, C.c_void_p(ids.data_ptr()), 0, None, None) == 0  # n == 0: no-op, even with no output
    assert lib.save_states(hp, None, 0, None, None) == 0
    assert lib.save_states(hp, C.c_void_p(ids.data_ptr()), 4, C.c_void_p(p + 16), None) == 0
    h.sync()
    with pytest.raises(ValueError):
        h.save_states(buf[1 : 1 + 4 * S], ids)  # misaligned rows are refused before the pointer crosses the ABI
    with pytest.raises(ValueError):
        h.save_states(buf[: 3 * S], ids)  # fewer rows than ids


def test_stream_order(cuda_lib, roms):
    import torch

    n = 96
    rom = roms("pokelike")
    a, b = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(cuda_lib, n, rom, 0)
    for h in (a, b):
        _mixed(h, n)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    g = torch.Generator(device="cuda").manual_seed(11)
    acts = [torch.randint(0, 8, (n,), generator=g, device="cuda", dtype=torch.uint8) for _ in range(3)]
    out_a = torch.zeros((n, S), dtype=torch.uint8, device="cuda")
    out_b = torch.zeros((n, S), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for t in range(3):
        a.run_action(acts[t], stream=s1.cuda_stream)
        a.save_states(out_a, stream=s2.cuda_stream)  # ordered after the step on the other stream by the handle
        b.run_action(acts[t], stream=s1.cuda_stream)
        b.save_states(out_b, stream=s1.cuda_stream)
        torch.cuda.synchronize()
        assert torch.equal(out_a, out_b), t
    assert np.array_equal(out_a.cpu().numpy(), _single(a, n))


def test_round_trip(cuda_lib, oracle_lib, roms):
    """Rows load back (gbenv_add_state_template + gbenv_load_template) into a fresh handle exactly as PyBoy's load_state would
    take them (the oracle): only STAT's mode bits 0-1, which a load keeps from the machine it lands on, may differ from the
    saved row; the restored emulator then steps like the source."""
    import torch

    n = 64
    rom = roms("pokelike")
    src = _capi.Handle(cuda_lib, n, rom, 0)
    _mixed(src, n)
    rng = np.random.default_rng(2)
    for _ in range(3):
        src.run_action(_dev(rng.integers(0, 8, n).astype(np.uint8)))
    rows = _gpu_rows(src, n)
    dst, ref = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    for i in range(n):
        for h in (dst, ref):
            h.load_template(h.add_state_template(rows[i].tobytes()), [i])
    again = _gpu_rows(dst, n)
    _first_diff(again, _cpu_rows(ref, n), "after load: oracle")
    stat = field_offsets(9)["lcd_regs"][0] + 4
    diff = again != rows
    assert not diff[:, np.arange(S) != stat].any(), "a reloaded row differs outside STAT"
    assert (((again[:, stat] ^ rows[:, stat]) & 0xFC) == 0).all()
    for t in range(20):
        act = rng.integers(0, 8, n).astype(np.uint8)
        src.run_action(_dev(act))
        dst.run_action(_dev(act))
        ref.run_action(act)
        if t in (0, 19):
            got = _gpu_rows(dst, n)
            _first_diff(got, _cpu_rows(ref, n), f"step {t}: oracle")
            _first_diff(got, _gpu_rows(src, n), f"step {t}: source")


def test_screen_field_is_the_packed_frame(cuda_lib, roms):
    import torch

    n = 45
    h = _capi.Handle(cuda_lib, n, roms("pokelike"), 0)
    _mixed(h, n)
    h.run_action(_dev(np.random.default_rng(4).integers(0, 8, n).astype(np.uint8)))
    ids = np.array([44, 0, 13, 13, 31, 32], np.int32)
    frames = torch.zeros((len(ids), _capi.FRAME_WORDS), dtype=torch.int32, device="cuda")
    h.capture_frames(frames, _dev(ids))
    rows = _gpu_rows(h, len(ids), ids)
    off, ln = field_offsets(9)["screen"]
    f = frames.cpu().numpy().view(np.uint32)
    px = np.arange(144 * 160)
    shades = (f[:, px >> 4] >> (2 * (px & 15)).astype(np.uint32)) & 3
    want = SHADE_WORDS[shades]
    got = np.ascontiguousarray(rows[:, off : off + ln]).view("<u4")
    assert np.array_equal(got, want)
    assert len(np.unique(shades)) > 1


def test_no_side_effects_on_a_vec_environment(cuda_lib, roms):
    import torch

    from pokegym_b200 import VecEnvironment

    n, mes = 80, 5
    blobs = [b.tobytes() for b in np.load(GOLDEN / "red_states_mixed.npz")["states"][:8]]
    vecs = [VecEnvironment(n, roms("pokelike"), blobs, max_episode_steps=mes, auto_reset=True) for _ in range(2)]
    outs = [v.reset()[0].clone() for v in vecs]
    assert torch.equal(outs[0], outs[1])
    g = torch.Generator(device="cuda").manual_seed(8)
    saved = 0
    for t in range(13):
        act = torch.randint(0, 8, (n,), generator=g, device="cuda", dtype=torch.uint8)
        rows = vecs[0].save_states(list(range(t % 3, n, 3)))
        saved += rows.shape[0]
        r0 = [x.clone() if torch.is_tensor(x) else x for x in vecs[0].step(act)[:3]]
        r1 = [x.clone() if torch.is_tensor(x) else x for x in vecs[1].step(act)[:3]]
        for a, b, what in zip(r0, r1, ("obs", "reward", "done")):
            assert torch.equal(a, b), (t, what)
        assert torch.equal(vecs[0].info(), vecs[1].info()), t
        full = vecs[0].save_states()
        assert full.shape == (n, S) and full.dtype == torch.uint8
        assert full[n - 1].cpu().numpy().tobytes() == vecs[0].save_state(n - 1)
    assert saved > 0
    torch.cuda.synchronize()
    a, b = vecs[0].save_states(), vecs[1].save_states()
    assert torch.equal(a, b)
    # the returned rows are .state files that load_state takes
    blob = a[17].cpu().numpy().tobytes()
    vecs[1].load_state(blob, [3])
    assert vecs[1].save_state(3)[: field_offsets(9)["lcd_regs"][0]] == blob[: field_offsets(9)["lcd_regs"][0]]
