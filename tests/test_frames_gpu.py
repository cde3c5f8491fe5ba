"""Batched frames on the device (gbenv_capture_frames / k_frames_capture, gbenv_frames_to_rgb / k_frames_to_rgb): bit-exact
against the CPU oracle and gbenv_screen, at scale, across streams, through VecEnvironment.screens and FrameRecorder (also
under PufferVecAdaptor), without side effects on the step, and their error paths."""
import numpy as np
import pytest

from pokegym_b200 import _capi

from test_frames_cpu import lcd_off_on

pytestmark = pytest.mark.gpu

FW = _capi.FRAME_WORDS


def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _gpu_frames(h, ids, n=None):
    import torch

    n = len(ids) if ids is not None else n
    out = torch.empty((n, FW), dtype=torch.int32, device="cuda")
    h.capture_frames(out, None if ids is None else _dev(np.asarray(ids, np.int32)))
    return out


def _gpu_decode(h, frames, channels):
    import torch

    out = torch.empty((len(frames), 144, 160, channels), dtype=torch.uint8, device="cuda")
    h.frames_to_rgb(frames, out, channels)
    return out.cpu().numpy()


def _cpu_frames(h, ids):
    out = np.zeros((len(ids), FW), np.uint32)
    h.capture_frames(out, np.ascontiguousarray(ids, np.int32))
    return out


def _cpu_screens(h, ids):
    return np.stack([h.screen(int(e)) for e in ids])


def _compare(gpu, cpu, ids, where, screen_sample=4):
    """CUDA packed frames == oracle packed frames; decoded RGB / grey == oracle_screen, and == gbenv_screen on a sample."""
    g = _gpu_frames(gpu, ids)
    packed = g.cpu().numpy().view(np.uint32)
    want = _cpu_frames(cpu, ids)
    assert np.array_equal(packed, want), f"{where}: packed frames differ from the oracle's"
    rgb, grey = _gpu_decode(gpu, g, 3), _gpu_decode(gpu, g, 1)
    screens = _cpu_screens(cpu, ids)
    assert np.array_equal(rgb, screens), f"{where}: decoded RGB differs from oracle_screen"
    assert np.array_equal(grey[..., 0], screens[..., 0]), f"{where}: decoded grey differs"
    for k in range(0, len(ids), max(1, len(ids) // screen_sample)):
        assert np.array_equal(rgb[k], gpu.screen(int(ids[k]))), f"{where}: decoded RGB differs from gbenv_screen (env {ids[k]})"
    return packed


@pytest.mark.parametrize("defer", ["1", "0"])
@pytest.mark.parametrize("rom_name,n", [("pokelike", 64), ("busy", 48), ("lcd_probe", 48), ("conformance", 56)])
def test_frames_match_oracle_after_every_entry_point(cuda_lib, oracle_lib, roms, monkeypatch, rom_name, n, defer):
    import torch

    monkeypatch.setenv("GBENV_DEFER", defer)  # read when the handle is created: 0 = lines drawn inside the emulation kernel
    rom = roms(rom_name)
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    rng = np.random.default_rng(17)

    def ids():  # any order, with duplicates
        return np.concatenate([rng.permutation(n), rng.integers(0, n, 9)]).astype(np.int32)

    for h in (gpu, cpu):
        h.tick(3, True)
    _compare(gpu, cpu, ids(), "tick")
    act = rng.integers(0, 8, n).astype(np.uint8)
    gpu.run_action(_dev(act))
    cpu.run_action(act)
    _compare(gpu, cpu, ids(), "run_action")
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    oc, rc, dc = np.zeros((n, _capi.OBS_BYTES), np.uint8), np.zeros(n), np.zeros(n, np.uint8)
    gpu.reset(og, max_episode_steps=6)
    cpu.reset(oc, max_episode_steps=6)
    _compare(gpu, cpu, ids(), "reset")
    distinct = set()
    for s in range(5):
        act = rng.integers(0, 8, n).astype(np.uint8)
        gpu.step(_dev(act), og, rg, dg)
        cpu.step(act, oc, rc, dc)
        distinct.update(f.tobytes() for f in _compare(gpu, cpu, ids(), f"step {s}"))
    skip = (rng.random(n) < 0.4).astype(np.uint8)
    act = rng.integers(0, 8, n).astype(np.uint8)
    gpu.step_masked(_dev(act), _dev(skip), og, rg, dg)
    cpu.step_masked(act, skip, oc, rc, dc)
    _compare(gpu, cpu, ids(), "step_masked")
    mask = (np.arange(n) % 3 == 0).astype(np.uint8)
    gpu.reset(og, mask=mask, max_episode_steps=6)
    cpu.reset(oc, mask=mask, max_episode_steps=6)
    _compare(gpu, cpu, ids(), "masked reset")
    for h in (gpu, cpu):
        lcd_off_on(h, n, lambda: None)
    _compare(gpu, cpu, ids(), "LCD off and on again")
    if rom_name != "conformance":  # that ROM leaves the screen blank
        assert len(distinct) > 1
    gpu.check()


@pytest.mark.parametrize("n", [4096, 32768])
def test_capture_at_scale(cuda_lib, roms, n):
    """All envs (NULL ids) and a scattered id list, against gbenv_screen on a sample of envs."""
    import torch

    gpu = _capi.Handle(cuda_lib, n, roms("pokelike"), 0)
    gpu.tick(30, True)
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    gpu.reset(og)
    gen = torch.Generator(device="cuda").manual_seed(n)
    for _ in range(4):
        gpu.step(torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8), og, rg, dg)
    rng = np.random.default_rng(n)
    sample = np.concatenate([[0, 31, 32, n - 1], rng.integers(0, n, 12)])
    full = _gpu_frames(gpu, None, n)
    rgb = _gpu_decode(gpu, full[torch.from_numpy(sample).cuda()].contiguous(), 3)
    for k, e in enumerate(sample):
        assert np.array_equal(rgb[k], gpu.screen(int(e))), e
    scattered = rng.permutation(n)[: n // 2].astype(np.int32)
    part = _gpu_frames(gpu, scattered)
    assert torch.equal(part, full[torch.from_numpy(scattered).long().cuda()])
    assert len({bytes(r) for r in full[:: n // 64].cpu().numpy()}) > 1


def test_capture_on_a_second_stream_sees_the_step(cuda_lib, oracle_lib, roms):
    """A capture queued on another torch stream right after a step on the default stream is ordered after that step."""
    import torch

    n = 1024
    rom = roms("busy")
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, 64, rom)
    for h in (gpu, cpu):
        h.tick(10, True)
    reps = n // 64
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    oc, rc, dc = np.zeros((64, _capi.OBS_BYTES), np.uint8), np.zeros(64), np.zeros(64, np.uint8)
    gpu.reset(og)
    cpu.reset(oc)
    side = torch.cuda.Stream()
    ids = _dev(np.arange(0, n, reps // 2 + 1, dtype=np.int32))
    frames = torch.empty((len(ids), FW), dtype=torch.int32, device="cuda")
    rng = np.random.default_rng(5)
    for s in range(4):
        act = rng.integers(0, 8, 64).astype(np.uint8)
        gpu.step(_dev(np.tile(act, reps)), og, rg, dg)  # default stream
        with torch.cuda.stream(side):
            gpu.capture_frames(frames, ids, stream=side.cuda_stream)
        cpu.step(act, oc, rc, dc)
        side.synchronize()
        want = _cpu_frames(cpu, ids.cpu().numpy() % 64)
        assert np.array_equal(frames.cpu().numpy().view(np.uint32), want), s


def _oracle_twin(oracle_lib, rom, n, mes):
    """The oracle driven as VecEnvironment drives the library: boot for 60 frames, reset all."""
    cpu = _capi.Handle(oracle_lib, n, rom)
    cpu.tick(60, True)
    obs = np.zeros((n, _capi.OBS_BYTES), np.uint8)
    cpu.reset(obs, max_episode_steps=mes)
    return cpu, obs


def _check_recorder(rec, packed_hist, done_hist, cpu):
    cap = rec.capacity
    want_p, want_d = np.stack(packed_hist[-cap:]), np.stack(done_hist[-cap:])
    assert rec.count == len(want_p)
    assert np.array_equal(rec.packed().cpu().numpy(), want_p), "packed frames differ from the oracle's, or out of order"
    assert np.array_equal(rec.dones().cpu().numpy(), want_d)
    n_ids = want_p.shape[1]
    decoded = np.zeros((len(want_p), n_ids, 144, 160, 3), np.uint8)
    cpu.frames_to_rgb(np.ascontiguousarray(want_p.reshape(-1, FW)), decoded.reshape(-1, 144, 160, 3), 3)
    assert np.array_equal(rec.frames().cpu().numpy(), decoded)
    assert np.array_equal(rec.frames(channels=1, start=2, stop=-1).cpu().numpy()[..., 0], decoded[2:-1, ..., 0])
    assert np.array_equal(rec.frames(start=-3).cpu().numpy(), decoded[-3:])


def test_recorder_follows_auto_reset_episodes(cuda_lib, oracle_lib, roms):
    """auto_reset with short episodes: every recorded frame is the oracle's screen after that step, before the oracle's
    reset of the envs that finished; the ring wraps and reads back oldest first."""
    import torch

    from pokegym_b200 import VecEnvironment

    n, mes, cap, steps = 40, 5, 7, 17
    rom = roms("pokelike")
    vec = VecEnvironment(n, rom, max_episode_steps=mes, auto_reset=True)
    vec.reset()
    ids = np.array([3, 0, 39, 17, 17, 8], np.int32)
    rec = vec.record_frames(ids, capacity=cap)
    assert vec.record_frames(ids, capacity=cap) is not rec and vec._recorder is not rec  # one recorder per VecEnvironment
    rec = vec.record_frames(ids, capacity=cap)
    cpu, oc = _oracle_twin(oracle_lib, rom, n, mes)
    rc, dc = np.zeros(n), np.zeros(n, np.uint8)
    rng = np.random.default_rng(9)
    packed, dones = [], []
    for s in range(steps):
        act = rng.integers(0, 8, n).astype(np.uint8)
        _, _, done, _, _ = vec.step(_dev(act))
        cpu.step(act, oc, rc, dc)
        packed.append(_cpu_frames(cpu, ids))
        dones.append(dc[ids].astype(bool))
        assert np.array_equal(done.cpu().numpy(), dc.astype(bool)), s
        if dc.any():
            cpu.reset(oc, mask=dc.copy(), max_episode_steps=mes)
        if s in (3, cap - 1, cap + 2):
            _check_recorder(rec, packed, dones, cpu)
    assert np.stack(dones).any()  # episodes ended while recording
    _check_recorder(rec, packed, dones, cpu)
    rec.clear()
    assert rec.count == 0 and rec.packed().shape == (0, len(ids), FW) and rec.frames().shape[0] == 0
    vec.step(_dev(np.zeros(n, np.uint8)))
    assert rec.count == 1
    assert vec.record_frames(None) is None
    vec.step(_dev(np.zeros(n, np.uint8)))
    assert rec.count == 1  # recording stopped
    vec.close()


def test_recorder_under_puffer_adaptor_records_skipped_envs(cuda_lib, oracle_lib, roms):
    """PufferVecAdaptor resets finished envs on the next send and makes them sit that step out: they record their unchanged
    frame and done False."""
    from pokegym_b200 import VecEnvironment
    from pokegym_b200.puffer import PufferVecAdaptor

    n, mes, cap, steps = 32, 4, 6, 14
    rom = roms("pokelike")
    vec = VecEnvironment(n, rom, max_episode_steps=mes)
    ids = np.array([5, 1, 30, 12], np.int32)
    rec = vec.record_frames(ids, capacity=cap)
    pv = PufferVecAdaptor(vec)
    pv.async_reset()
    cpu, oc = _oracle_twin(oracle_lib, rom, n, mes)
    rc, dc = np.zeros(n), np.zeros(n, np.uint8)
    pending = np.zeros(n, np.uint8)
    rng = np.random.default_rng(21)
    packed, dones = [], []
    skipped = 0
    for s in range(steps):
        act = rng.integers(0, 8, n).astype(np.uint8)
        pv.send(_dev(act))
        pv.recv()
        if pending.any():
            cpu.reset(oc, mask=pending.copy(), max_episode_steps=mes)
            cpu.step_masked(act, pending.copy(), oc, rc, dc)
            skipped += int(pending[ids].sum())
        else:
            cpu.step(act, oc, rc, dc)
        packed.append(_cpu_frames(cpu, ids))
        dones.append(dc[ids].astype(bool))
        pending = dc.copy()
    assert skipped
    _check_recorder(rec, packed, dones, cpu)
    vec.close()


def test_recorder_has_no_side_effects(cuda_lib, roms):
    """200 steps with and without a recorder: byte-identical obs, rewards, dones and info rows."""
    import torch

    from pokegym_b200 import VecEnvironment

    n, mes = 128, 30
    rom = roms("pokelike")
    plain = VecEnvironment(n, rom, max_episode_steps=mes, auto_reset=True)
    recorded = VecEnvironment(n, rom, max_episode_steps=mes, auto_reset=True)
    rec = recorded.record_frames(np.arange(0, n, 8), capacity=50)
    for v in (plain, recorded):
        v.reset()
    gen = torch.Generator(device="cuda").manual_seed(7)
    for s in range(200):
        act = torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8)
        a = plain.step(act)
        b = recorded.step(act)
        for x, y in zip(a[:3], b[:3]):
            assert torch.equal(x, y), s
        if s % 20 == 19:
            assert torch.equal(plain.info(), recorded.info()), s
    assert rec.count == 50 and bool(rec.dones().any())
    assert torch.equal(plain.info(), recorded.info())
    plain.close()
    recorded.close()


def test_screens_and_error_paths(cuda_lib, roms):
    import torch

    from pokegym_b200 import VecEnvironment

    n = 40
    vec = VecEnvironment(n, roms("pokelike"))
    vec.reset()
    vec.step(torch.zeros(n, dtype=torch.uint8, device="cuda"))
    allrgb = vec.screens()
    assert allrgb.shape == (n, 144, 160, 3) and allrgb.dtype == torch.uint8 and allrgb.device.type == "cuda"
    for e in (0, 13, n - 1):
        assert np.array_equal(allrgb[e].cpu().numpy(), vec.handle.screen(e))
    ids = [7, 2, 7]
    grey = vec.screens(ids, channels=1)
    assert grey.shape == (3, 144, 160, 1)
    assert torch.equal(grey[..., 0], allrgb[ids, ..., 0])
    out = torch.empty((3, 144, 160, 3), dtype=torch.uint8, device="cuda")
    assert vec.screens(torch.tensor(ids, device="cuda"), out=out).data_ptr() == out.data_ptr()
    assert torch.equal(out, allrgb[ids])
    with pytest.raises(ValueError):
        vec.screens(channels=2)
    for bad in ([n], [-1], [], [[0]]):
        with pytest.raises(ValueError):
            vec.screens(bad)
    for bad_out in (torch.empty((3, 144, 160, 1), dtype=torch.uint8, device="cuda"), torch.empty((3, 144, 160, 3), dtype=torch.int32, device="cuda"),
                    torch.empty((3, 144, 160, 3), dtype=torch.uint8)):
        with pytest.raises(ValueError):
            vec.screens(ids, out=bad_out)
    size = 3 * 144 * 160 * 3
    misaligned = torch.empty(size + 16, dtype=torch.uint8, device="cuda")[1:1 + size].view(3, 144, 160, 3)
    with pytest.raises(ValueError, match="aligned"):
        vec.screens(ids, out=misaligned)
    frames = torch.empty((1, FW), dtype=torch.int32, device="cuda")
    with pytest.raises(_capi.GbEnvError, match="bad argument"):  # the library checks the alignment too
        vec.handle.frames_to_rgb(frames, misaligned[:1], 3)
    with pytest.raises(_capi.GbEnvError, match="bad argument"):
        vec.handle.frames_to_rgb(frames, out[:1], 2)
    # ids are bounds-checked on the device too: the rows of out-of-range ids stay as they were
    rows = torch.full((4, FW), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    vec.handle.capture_frames(rows, torch.tensor([1, -5, n, 2], dtype=torch.int32, device="cuda"))
    assert bool((rows[1:3] == 0x5A5A5A5A).all())
    assert torch.equal(rows[[0, 3]], _gpu_frames(vec.handle, [1, 2]))
    with pytest.raises(ValueError):
        vec.record_frames([0, 1], capacity=0)
    with pytest.raises(ValueError):
        vec.record_frames([0, 1])
    with pytest.raises(ValueError):
        vec.record_frames([0, n], capacity=4)
    vec.close()
