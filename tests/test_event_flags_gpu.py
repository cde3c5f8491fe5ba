"""Event flags on the device (gbenv_event_flags / k_event_flags): bit-exact against the CPU oracle after every entry point,
at full batch size, pinned to the reference's recorded info dicts, through VecEnvironment.episode_infos / event_counts /
full_info, EnvGroups and PufferVecAdaptor(full_infos=True), across streams, and its error paths."""
import ctypes as C

import numpy as np
import pytest

from helpers import GOLDEN, info_fingerprint
from pokegym_b200 import _capi
from pokegym_b200 import info as I
from test_event_flags_cpu import RECORDINGS, randomise_wram, replay_info_steps

pytestmark = pytest.mark.gpu

EW = _capi.EVENT_WORDS


def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _gpu_flags(h, ids, n=None):
    import torch

    n = len(ids) if ids is not None else n
    out = torch.zeros((n, EW), dtype=torch.int32, device="cuda")
    h.event_flags(out, None if ids is None else _dev(np.asarray(ids, np.int32)))
    return out.cpu().numpy().view(np.uint32)


def _cpu_flags(h, ids=None, n=None):
    n = len(ids) if ids is not None else n
    out = np.zeros((n, EW), np.uint32)
    h.event_flags(out, None if ids is None else np.ascontiguousarray(ids, np.int32))
    return out


def _compare(gpu, cpu, n, rng, where):
    want = _cpu_flags(cpu, n=n)
    assert np.array_equal(_gpu_flags(gpu, None, n), want), f"{where}: NULL ids"
    ids = np.concatenate([rng.permutation(n), rng.integers(0, n, 9)]).astype(np.int32)
    assert np.array_equal(_gpu_flags(gpu, ids), want[ids]), f"{where}: permuted / duplicated ids"
    import torch

    bad = np.array([n - 1, -3, n, 0, 1 << 30], np.int32)
    rows = torch.full((len(bad), EW), 0x3C3C3C3C, dtype=torch.int32, device="cuda")
    gpu.event_flags(rows, _dev(bad))
    rows = rows.cpu().numpy().view(np.uint32)
    assert (rows[[1, 2, 4]] == 0x3C3C3C3C).all(), f"{where}: a row of an out-of-range id was written"
    assert np.array_equal(rows[[0, 3]], want[[n - 1, 0]]), where
    return want


@pytest.mark.parametrize("lanes", [1, 32])
@pytest.mark.parametrize("rom_name,n", [("pokelike", 64), ("conformance", 56)])
def test_event_flags_match_oracle_after_every_entry_point(cuda_lib, oracle_lib, roms, rom_name, n, lanes):
    import torch

    rom = roms(rom_name)
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    gpu.set_lanes_per_warp(lanes)
    rng = np.random.default_rng(23 + lanes)
    for h in (gpu, cpu):
        h.tick(3, True)
    _compare(gpu, cpu, n, rng, "tick")
    data = rng.integers(0, 256, (n, 0x200), dtype=np.uint8)
    for h in (gpu, cpu):
        for e in range(n):
            h.write_mem(e, 0xD700, data[e])
    first = _compare(gpu, cpu, n, rng, "random WRAM")
    assert first.any() and len({r.tobytes() for r in first}) > n // 2
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    oc, rc, dc = np.zeros((n, _capi.OBS_BYTES), np.uint8), np.zeros(n), np.zeros(n, np.uint8)
    gpu.reset(og, max_episode_steps=4)
    cpu.reset(oc, max_episode_steps=4)
    _compare(gpu, cpu, n, rng, "reset")
    finished = 0
    for s in range(9):
        act = rng.integers(0, 8, n).astype(np.uint8)
        if s == 5:
            skip = (rng.random(n) < 0.4).astype(np.uint8)
            gpu.step_masked(_dev(act), _dev(skip), og, rg, dg)
            cpu.step_masked(act, skip, oc, rc, dc)
            where = "step_masked"
        else:
            gpu.step(_dev(act), og, rg, dg)
            cpu.step(act, oc, rc, dc)
            where = f"step {s}"
        assert np.array_equal(dg.cpu().numpy(), dc), where
        _compare(gpu, cpu, n, rng, where)
        if dc.any():  # auto-reset on the device, masked by the done vector the step wrote
            gpu.reset_dev(og, mask_dev=dg, max_episode_steps=4)
            cpu.reset(oc, mask=dc.copy(), max_episode_steps=4)
            finished += int(dc.sum())
            _compare(gpu, cpu, n, rng, f"auto-reset after step {s}")
    assert finished
    gpu.check()


@pytest.mark.parametrize("n", [4096, 32768])
def test_full_size_batch_matches_replicated_small_batch(cuda_lib, oracle_lib, roms, n):
    """Env i starts from the state of oracle env i mod 64 (random event WRAM) and gets its actions: every row of flags, and
    the counts, equal the 64-env oracle's replicated."""
    import torch

    from pokegym_b200.vec_env import event_counts_from_flags

    base, reps = 64, n // 64
    rom = roms("pokelike")
    cpu = _capi.Handle(oracle_lib, base, rom)
    cpu.tick(30, False)
    randomise_wram(cpu, base, seed=n)
    gpu = _capi.Handle(cuda_lib, n, rom, 0)
    for e in range(base):
        blob = cpu.save_state(e)
        for h, ids in ((gpu, np.arange(e, n, base)), (cpu, [e])):
            h.set_initial_template(h.add_state_template(blob), np.asarray(ids, np.int32))
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    oc, rc, dc = np.zeros((base, _capi.OBS_BYTES), np.uint8), np.zeros(base), np.zeros(base, np.uint8)
    gpu.reset(og, max_episode_steps=50)
    cpu.reset(oc, max_episode_steps=50)
    rng = np.random.default_rng(n)
    for s in range(3):
        act = rng.integers(0, 8, base).astype(np.uint8)
        gpu.step(_dev(np.tile(act, reps)), og, rg, dg)
        cpu.step(act, oc, rc, dc)
    want = _cpu_flags(cpu, n=base)
    assert want.any()
    full = torch.empty((n, EW), dtype=torch.int32, device="cuda")
    gpu.event_flags(full)
    assert bool((full.view(reps, base, EW) == _dev(want.view(np.int32))[None]).all())
    ids = rng.permutation(n)[: n // 3].astype(np.int32)
    assert np.array_equal(_gpu_flags(gpu, ids), want[ids % base])
    counts = event_counts_from_flags(torch, full, None, torch.empty(130, dtype=torch.int64, device="cuda"))
    assert np.array_equal(counts.cpu().numpy(), reps * I.unpack_event_words(want).sum(0))


@pytest.mark.parametrize("name", RECORDINGS)
def test_info_from_cuda_event_flags_matches_the_reference(cuda_lib, roms, name):
    """A 1-env handle replays the reference's recording; at each step with an info dict, the dict built from
    Handle.event_flags + get_info + counts_map has the recorded fingerprint."""
    import torch

    gold = np.load(GOLDEN / f"ref_wrapper_{name}.npz")
    h = _capi.Handle(cuda_lib, 1, roms(str(gold["rom_name"])), 0)
    flags = torch.zeros((1, EW), dtype=torch.int32, device="cuda")
    seen = 0
    for i, row, want in replay_info_steps(h, gold, to_dev=lambda a: torch.from_numpy(a).cuda(), to_host=lambda t: t.cpu().numpy()):
        h.event_flags(flags)
        mine = I.build_info_from_events(row, I.unpack_event_words(flags)[0], counts_map=h.counts_map(0))
        assert info_fingerprint(mine) == want, f"step {i}: info dict differs from the reference's"
        seen += 1
    assert seen == len(gold["info_steps"])


def _without_map(d):
    d = dict(d, pokemon_exploration_map=None)
    d["stats"] = dict(d["stats"], pokemon_exploration_map=None)
    return d


def _old_full_info(vec, e):
    """full_info as it was built before gbenv_event_flags: bus reads of the env's WRAM and build_info."""
    row = vec.info()[e].cpu().numpy()
    wram = vec.handle.read_mem(e, 0xD700, 0x200)
    return I.build_info(row, lambda a: int(wram[a - 0xD700]), counts_map=vec.handle.counts_map(e).astype(np.float64), reward_scale=vec.reward_scale)


@pytest.mark.parametrize("auto_reset", [False, True])
def test_episode_infos_equal_full_info(cuda_lib, roms, auto_reset):
    import torch

    from pokegym_b200 import VecEnvironment

    n, mes = 48, 6
    vec = VecEnvironment(n, roms("pokelike"), max_episode_steps=mes, auto_reset=auto_reset)
    vec.reset()
    randomise_wram(vec.handle, n, seed=11)
    gen = torch.Generator(device="cuda").manual_seed(3)
    checked = 0
    for s in range(2 * mes + 1):
        act = torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8)
        _, _, done, _, _ = vec.step(act)
        ended = np.nonzero(done.cpu().numpy())[0]
        got = vec.episode_infos(done)
        assert list(got) == list(ended), s
        for e in ended:
            full = vec.full_info(int(e))
            assert got[e] == _without_map(full), (s, e)
            old = _old_full_info(vec, int(e))
            assert np.array_equal(full["pokemon_exploration_map"], old["pokemon_exploration_map"])
            assert _without_map(full) == _without_map(old), (s, e)
            checked += 1
        if not auto_reset and len(ended):
            vec.reset(mask=done)
    assert checked >= n
    assert vec.episode_infos(torch.zeros(n, dtype=torch.bool, device="cuda")) == {}
    some = [0, 7, n - 1]
    mask = np.zeros(n, np.uint8)
    mask[some] = 1
    assert list(vec.episode_infos(mask)) == some
    vec.close()


def test_event_counts_match_oracle_and_env_groups(cuda_lib, oracle_lib, roms):
    import torch

    from pokegym_b200 import VecEnvironment
    from pokegym_b200.groups import EnvGroups

    n, mes = 80, 5
    rom = roms("pokelike")
    vec = VecEnvironment(n, rom, max_episode_steps=mes)
    cpu = _capi.Handle(oracle_lib, n, rom)  # driven as VecEnvironment drives the library
    cpu.tick(60, True)
    oc, rc, dc = np.zeros((n, _capi.OBS_BYTES), np.uint8), np.zeros(n), np.zeros(n, np.uint8)
    vec.reset(max_episode_steps=mes)
    cpu.reset(oc, max_episode_steps=mes)
    data = randomise_wram(cpu, n, seed=8)
    for e in range(n):
        vec.handle.write_mem(e, 0xD700, data[e])
    rng = np.random.default_rng(8)
    for s in range(mes):
        act = rng.integers(0, 8, n).astype(np.uint8)
        _, _, done, _, _ = vec.step(_dev(act))
        cpu.step(act, oc, rc, dc)
    assert dc.all() and np.array_equal(done.cpu().numpy(), dc.astype(bool))
    bits = I.unpack_event_words(_cpu_flags(cpu, n=n)).astype(np.int64)
    rand = rng.random(n) < 0.5
    out = torch.empty(130, dtype=torch.int64, device="cuda")
    for mask, m in ((None, np.ones(n, bool)), (done, dc.astype(bool)), (_dev(rand.astype(np.uint8)), rand), (np.zeros(n, np.uint8), np.zeros(n, bool))):
        got = vec.event_counts(mask)
        assert got.dtype == torch.int64 and got.device.type == "cuda"
        assert np.array_equal(got.cpu().numpy(), bits[m].sum(0))
        assert vec.event_counts(mask, out=out) is out and torch.equal(out, got)
    with pytest.raises(ValueError):
        vec.event_counts(out=torch.empty(130, dtype=torch.int32, device="cuda"))
    groups = EnvGroups(cuda_lib, 2 * n, rom, n_groups=4)
    single = _capi.Handle(cuda_lib, 2 * n, rom, 0)
    for h in (*groups.handles, single):
        h.tick(3, True)
    big = np.concatenate([data, data[::-1]])
    for e in range(2 * n):
        single.write_mem(e, 0xD700, big[e])
        groups.handles[e // (n // 2)].write_mem(e % (n // 2), 0xD700, big[e])
    flags = torch.empty((2 * n, EW), dtype=torch.int32, device="cuda")
    single.event_flags(flags)
    from pokegym_b200.vec_env import event_counts_from_flags

    mask = _dev((rng.random(2 * n) < 0.5).astype(np.uint8))
    for m in (None, mask):
        want = event_counts_from_flags(torch, flags, m, torch.empty(130, dtype=torch.int64, device="cuda"))
        got = groups.event_counts(torch.empty(130, dtype=torch.int64, device="cuda"), m)
        assert torch.equal(got, want)
    assert int(want.sum()) > 0
    groups.close()
    vec.close()


def test_puffer_adaptor_full_infos(cuda_lib, roms):
    """full_infos=True: at each step the dicts of exactly the envs whose done is set, equal to episode_infos.  The default
    adaptor, stepped with the same actions, delivers the info_row_to_dict rows as before."""
    from pokegym_b200 import VecEnvironment
    from pokegym_b200.puffer import PufferVecAdaptor

    n, mes = 36, 4
    rom = roms("pokelike")
    full = PufferVecAdaptor(VecEnvironment(n, rom, max_episode_steps=mes), full_infos=True)
    plain = PufferVecAdaptor(VecEnvironment(n, rom, max_episode_steps=mes))
    for pv in (full, plain):
        pv.async_reset()
        randomise_wram(pv.vec.handle, n, seed=4)
    rng = np.random.default_rng(4)
    delivered = 0
    for s in range(12):
        act = rng.integers(0, 8, n).astype(np.uint8)
        for pv in (full, plain):
            pv.send(_dev(act))
        _, _, d_full, _, infos_full, _, _ = full.recv()
        _, _, d_plain, _, infos_plain, _, _ = plain.recv()
        assert np.array_equal(d_full.cpu().numpy(), d_plain.cpu().numpy()), s
        ended = np.nonzero(d_full.cpu().numpy())[0]
        assert len(infos_full) == len(infos_plain) == len(ended), s
        assert infos_full == list(full.vec.episode_infos(d_full).values()), s
        rows = plain.vec.info().cpu().numpy()
        assert infos_plain == [I.info_row_to_dict(rows[e]) for e in ended], s
        for d in infos_full:
            assert d["pokemon_exploration_map"] is None and "gym_events" in d and "detailed_rewards_dojo" in d
        delivered += len(infos_full)
    assert delivered
    full.vec.close()
    plain.vec.close()


def test_event_flags_on_a_second_stream_see_the_step(cuda_lib, oracle_lib, roms):
    """The reset that loads every env's save-state (new event flags) and a step are queued on the default stream; event_flags
    queued right after on another torch stream sees them."""
    import torch

    base, n = 64, 2048
    rom = roms("pokelike")
    cpu = _capi.Handle(oracle_lib, base, rom)
    cpu.tick(10, True)
    randomise_wram(cpu, base, seed=1)
    gpu = _capi.Handle(cuda_lib, n, rom, 0)
    gpu.tick(10, True)
    for e in range(base):
        blob = cpu.save_state(e)
        for h, ids in ((gpu, np.arange(e, n, base)), (cpu, [e])):
            h.set_initial_template(h.add_state_template(blob), np.asarray(ids, np.int32))
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    oc, rc, dc = np.zeros((base, _capi.OBS_BYTES), np.uint8), np.zeros(base), np.zeros(base, np.uint8)
    side = torch.cuda.Stream()
    flags = torch.zeros((n, EW), dtype=torch.int32, device="cuda")
    act = np.random.default_rng(2).integers(0, 8, base).astype(np.uint8)
    acts = _dev(np.tile(act, n // base))
    gpu.reset_dev(og)  # default stream
    gpu.step(acts, og, rg, dg)
    with torch.cuda.stream(side):
        gpu.event_flags(flags, stream=side.cuda_stream)
    side.synchronize()
    cpu.reset(oc)
    cpu.step(act, oc, rc, dc)
    want = _cpu_flags(cpu, n=base)
    assert want.any()
    assert np.array_equal(flags.cpu().numpy().view(np.uint32), np.tile(want, (n // base, 1)))


def test_event_flags_argument_errors(cuda_lib, roms):
    import torch

    from pokegym_b200 import VecEnvironment

    n = 40
    vec = VecEnvironment(n, roms("pokelike"))
    vec.reset()
    h, lib = vec.handle, cuda_lib
    out = torch.zeros((n + 1, EW), dtype=torch.int32, device="cuda")
    ids = torch.zeros(4, dtype=torch.int32, device="cuda")
    p_out, p_ids = C.c_void_p(out.data_ptr()), C.c_void_p(ids.data_ptr())
    assert lib.event_flags(None, p_ids, 4, p_out, None) == -1  # GBENV_E_ARG
    assert lib.event_flags(h._h, p_ids, 4, None, None) == -1
    assert lib.event_flags(h._h, p_ids, -1, p_out, None) == -1
    assert lib.event_flags(h._h, None, n + 1, p_out, None) == -1
    assert lib.event_flags(h._h, p_ids, 4, C.c_void_p(out.data_ptr() + 2), None) == -1  # misaligned
    assert lib.event_flags(h._h, p_ids, 0, p_out, None) == 0
    assert lib.event_flags(h._h, None, 0, None, None) == 0
    torch.cuda.synchronize()
    assert not bool(out.any())
    with pytest.raises(ValueError):
        h.event_flags(out[:1], ids)
    with pytest.raises(_capi.GbEnvError, match="bad argument"):
        h.event_flags(out)
    for bad in ([n], [-1], [], [[0]]):
        with pytest.raises(ValueError):
            vec.event_flags(bad)
    with pytest.raises(ValueError):
        vec.event_flags([1, 2], out=torch.zeros((2, EW), dtype=torch.int64, device="cuda"))
    mine = vec.event_flags([3, 3, 0])
    assert mine.shape == (3, EW) and mine.dtype == torch.int32 and torch.equal(mine, vec.event_flags()[[3, 3, 0]])
    vec.close()
