"""Episode-end reductions on the device: the heat-map sum (gbenv_counts_map_sum / k_cm_sum) and the masked info sum
(gbenv_reduce_info_masked), against the CPU oracle, through VecEnvironment and EnvGroups, and their error paths."""
import numpy as np
import pytest

from pokegym_b200 import _capi

pytestmark = pytest.mark.gpu

MAP_SHAPE = (_capi.COUNTS_H, _capi.COUNTS_W)


def _map_sum(h, mask=None):
    import torch

    out = torch.full(MAP_SHAPE, 7, dtype=torch.int64, device="cuda")  # overwritten, not accumulated into
    h.counts_map_sum(out, None if mask is None else torch.from_numpy(np.ascontiguousarray(mask, np.uint8)).cuda())
    return out.cpu().numpy()


def _oracle_map_sum(h, mask=None):
    out = np.zeros(MAP_SHAPE, np.int64)
    h.counts_map_sum(out, None if mask is None else np.ascontiguousarray(mask, np.uint8))
    return out


def _info_sum(h, mask=None):
    import torch

    out = torch.zeros(_capi.INFO_SCALARS, dtype=torch.float64, device="cuda")
    h.reduce_info_masked(out, None if mask is None else torch.from_numpy(np.ascontiguousarray(mask, np.uint8)).cuda())
    return out.cpu().numpy()


def _oracle_info_sum(h, mask=None):
    out = np.zeros(_capi.INFO_SCALARS)
    h.reduce_info_masked(out, None if mask is None else np.ascontiguousarray(mask, np.uint8))
    return out


def test_map_sum_and_masked_info_match_oracle_through_many_maps(cuda_lib, oracle_lib, roms):
    """48 envs, three of them teleported through a new map and all four 64-row bands every step (their maps hold many
    blocks and the -1 marks of map transitions); the even envs finish at step 36, the odd ones are reset at step 30.  The
    map sum is exactly the oracle's for the masks NULL / done / random / zeros; the masked info sum is compared before the
    masked envs are reset (the oracle zeroes a row on reset, the CUDA library keeps the row of the last step)."""
    import torch

    n, steps, mes = 48, 56, 36
    rom = roms("pokelike")
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    oc, rc, dc = np.zeros((n, _capi.OBS_BYTES), np.uint8), np.zeros(n), np.zeros(n, np.uint8)
    gpu.tick(40, True)
    cpu.tick(40, True)
    gpu.reset(og, max_episode_steps=mes)
    cpu.reset(oc, max_episode_steps=mes)
    rng = np.random.default_rng(11)
    odd = (np.arange(n) % 2).astype(np.uint8)
    checked = 0
    for s in range(steps):
        if s == 30:
            assert np.allclose(_info_sum(gpu, odd), _oracle_info_sum(cpu, odd), rtol=1e-12, atol=0)
            gpu.reset(og, mask=odd, max_episode_steps=mes)
            cpu.reset(oc, mask=odd, max_episode_steps=mes)
            assert np.array_equal(_map_sum(gpu), _oracle_map_sum(cpu)), "a reset changed the heat maps"
        for k, e in enumerate((1, 17, 40)):
            m, r, c = (7 * s + 31 * k) % 248, (37 * s + 5 * k) % 250, (11 * s + 3 * k) % 250
            for h in (gpu, cpu):
                h.write_mem(e, 0xD35E, [m])
                h.write_mem(e, 0xD361, [r])
                h.write_mem(e, 0xD362, [c])
        act = rng.integers(0, 8, n).astype(np.uint8)
        gpu.step(torch.from_numpy(act).cuda(), og, rg, dg)
        cpu.step(act, oc, rc, dc)
        assert np.array_equal(dg.cpu().numpy(), dc), s
        if s in (0, 9, 35, steps - 1):
            rand = (rng.random(n) < 0.5).astype(np.uint8)
            for mask in (None, dc.copy(), rand, np.zeros(n, np.uint8)):
                want = _oracle_map_sum(cpu, mask)
                got = _map_sum(gpu, mask)
                assert np.array_equal(got, want), (s, None if mask is None else int(mask.sum()))
                assert np.allclose(_info_sum(gpu, mask), _oracle_info_sum(cpu, mask), rtol=1e-12, atol=0), s
            checked += 1
    assert dc[::2].all() and not dc[1::2].any()
    full = _oracle_map_sum(cpu)
    assert (full < 0).any() and (full > 0).sum() > 100  # the maps the sums ran over are not trivial
    assert _info_sum(gpu, np.zeros(n, np.uint8)).sum() == 0
    assert np.array_equal(_info_sum(gpu), _info_sum(gpu, np.ones(n, np.uint8)))
    gpu.check()
    assert checked == 4


@pytest.mark.parametrize("n,steps", [(4096, 40), (32768, 6)])
def test_map_sum_of_replicated_batch(cuda_lib, oracle_lib, roms, n, steps):
    """Env i plays env i mod 64, so every sum is reps times the 64-env oracle's.  At these sizes the grid has several env
    chunks, each adding its partial sums into the result."""
    import torch

    base = 64
    reps = n // base
    rom = roms("pokelike")
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, base, rom)
    gpu.tick(30, False)
    cpu.tick(30, False)
    og = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rg = torch.zeros(n, dtype=torch.float64, device="cuda")
    dg = torch.zeros(n, dtype=torch.uint8, device="cuda")
    oc, rc, dc = np.zeros((base, _capi.OBS_BYTES), np.uint8), np.zeros(base), np.zeros(base, np.uint8)
    gpu.reset(og)
    cpu.reset(oc)
    rng = np.random.default_rng(8)
    for _ in range(steps):
        act = rng.integers(0, 8, base).astype(np.uint8)
        gpu.step(torch.from_numpy(np.tile(act, reps)).cuda(), og, rg, dg)
        cpu.step(act, oc, rc, dc)
    gpu.check()
    mask = (rng.random(base) < 0.5).astype(np.uint8)
    want = _oracle_map_sum(cpu)
    assert (want != 0).sum() > 10  # the 64 envs start on one cell; a few steps spread them over some
    assert np.array_equal(_map_sum(gpu), reps * want)
    assert np.array_equal(_map_sum(gpu, np.tile(mask, reps)), reps * _oracle_map_sum(cpu, mask))
    tail = np.zeros(n, np.uint8)
    tail[-base:] = 1  # only the last chunk contributes
    assert np.array_equal(_map_sum(gpu, tail), want)
    assert np.allclose(_info_sum(gpu, np.tile(mask, reps)), reps * _oracle_info_sum(cpu, mask), rtol=1e-12, atol=0)


def test_vec_environment_sums_over_finished_episodes(cuda_lib, roms):
    """VecEnvironment(auto_reset=True) resets finished envs inside step(); their info rows are still those of their last
    step, so info_sum(mask=done) is the sum over the episodes that just ended."""
    import torch

    from pokegym_b200 import VecEnvironment

    n, mes = 96, 6
    vec = VecEnvironment(n, roms("pokelike"), max_episode_steps=mes, auto_reset=True)
    vec.reset()
    short = np.zeros(n, np.uint8)
    short[: n // 3] = 1
    vec.reset(mask=short, max_episode_steps=4)  # staggered episodes: some steps finish only part of the batch
    vec.max_episode_steps = mes
    g = torch.Generator(device="cuda").manual_seed(3)
    partial = 0
    for t in range(14):
        obs, rew, done, _, _ = vec.step(torch.randint(0, 8, (n,), generator=g, device="cuda", dtype=torch.uint8))
        s = vec.info_sum(mask=done)
        rows = vec.info()
        assert torch.allclose(s, rows[done].sum(dim=0), rtol=1e-12, atol=0), t
        k = int(done.sum())
        assert s[0].item() == k  # slot 0: the number of episodes that ended
        if k:
            assert bool((rows[done][:, 1] >= 4).all())  # "step" of the finished episode, not a row cleared by the reset
            m = vec.exploration_map_sum(mask=done)
            assert m.dtype == torch.int64 and tuple(m.shape) == MAP_SHAPE
            want = sum(vec.handle.counts_map(e).astype(np.int64) for e in torch.nonzero(done).flatten().tolist())
            assert np.array_equal(m.cpu().numpy(), want), t
            partial += k < n
    assert partial  # at least one step where only some envs finished
    assert torch.equal(vec.info_sum(), vec.info_sum(mask=torch.ones(n, dtype=torch.bool, device="cuda")))
    out = torch.empty(MAP_SHAPE, dtype=torch.int64, device="cuda")
    assert vec.exploration_map_sum(out=out).data_ptr() == out.data_ptr()
    assert np.array_equal(out.cpu().numpy(), sum(vec.handle.counts_map(e).astype(np.int64) for e in range(n)))
    assert not vec.exploration_map_sum(mask=[0] * n).any()  # an array-like mask
    with pytest.raises(ValueError):
        vec.exploration_map_sum(mask=np.ones(n + 1, np.uint8))
    with pytest.raises(ValueError):
        vec.info_sum(mask=torch.ones(n - 1, dtype=torch.bool, device="cuda"))
    with pytest.raises(ValueError):
        vec.exploration_map_sum(out=torch.empty(MAP_SHAPE, dtype=torch.int32, device="cuda"))
    vec.close()


def test_env_groups_sums_equal_one_handle(cuda_lib, roms):
    import torch

    from pokegym_b200 import EnvGroups

    E, G = 128, 2
    rom = roms("pokelike")
    groups = EnvGroups(cuda_lib, E, rom, n_groups=G)
    groups.for_each(lambda h, g, st: h.tick(60, True, stream=st))
    one = _capi.Handle(cuda_lib, E, rom, 0)
    one.tick(60, True)
    dev = groups.device
    obs, obs1 = (torch.zeros((E, _capi.OBS_BYTES), dtype=torch.uint8, device=dev) for _ in range(2))
    rew, rew1 = (torch.zeros(E, dtype=torch.float64, device=dev) for _ in range(2))
    done, done1 = (torch.zeros(E, dtype=torch.uint8, device=dev) for _ in range(2))
    groups.reset(obs, max_episode_steps=5)
    one.reset(obs1, max_episode_steps=5)
    rng = np.random.default_rng(2)
    for t in range(5):
        act = torch.from_numpy(rng.integers(0, 8, E).astype(np.uint8)).to(dev)
        groups.step(act, obs, rew, done, join=True)
        one.step(act, obs1, rew1, done1)
    torch.cuda.synchronize()
    assert torch.equal(done, done1) and bool(done.all())
    mask = torch.from_numpy((rng.random(E) < 0.5).astype(np.uint8)).to(dev)
    mask[E // G - 1], mask[E // G] = 1, 0  # both sides of the group boundary
    for m in (None, mask, mask.bool()):
        s_g, s_1 = torch.zeros(_capi.INFO_SCALARS, dtype=torch.float64, device=dev), torch.zeros(_capi.INFO_SCALARS, dtype=torch.float64, device=dev)
        groups.reduce_info(s_g, mask=m)
        one.reduce_info_masked(s_1, None if m is None else mask)
        assert torch.allclose(s_g, s_1, rtol=1e-12, atol=0)  # partial sums per group: the association differs
        m_g, m_1 = torch.empty(MAP_SHAPE, dtype=torch.int64, device=dev), torch.empty(MAP_SHAPE, dtype=torch.int64, device=dev)
        groups.exploration_map_sum(m_g, mask=m)
        one.counts_map_sum(m_1, None if m is None else mask)
        assert torch.equal(m_g, m_1)
        assert bool((m_1 != 0).any())
    with pytest.raises(ValueError):
        groups.exploration_map_sum(m_g, mask=torch.ones(E - 1, dtype=torch.uint8, device=dev))
    groups.close()


def test_map_sum_error_paths(cuda_lib, roms, monkeypatch):
    import torch

    rom = roms("pokelike")
    out = torch.empty(MAP_SHAPE, dtype=torch.int64, device="cuda")
    h = _capi.Handle(cuda_lib, 4, rom)
    with pytest.raises(_capi.GbEnvError, match="bad argument"):
        h.counts_map_sum(None)
    monkeypatch.setenv("GBENV_COUNTS_MAP", "0")
    off = _capi.Handle(cuda_lib, 4, rom)
    with pytest.raises(_capi.GbEnvError, match="exploration map tracking is disabled"):
        off.counts_map_sum(out)
    monkeypatch.delenv("GBENV_COUNTS_MAP")
    # a heat-map pool that runs dry: once check() has seen it, the sum over the now incomplete maps is refused
    n = 48
    monkeypatch.setenv("GBENV_COUNTS_BLOCKS", "50")
    tiny = _capi.Handle(cuda_lib, n, rom)
    tiny.tick(40, True)
    obs = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
    rew = torch.zeros(n, dtype=torch.float64, device="cuda")
    done = torch.zeros(n, dtype=torch.uint8, device="cuda")
    tiny.reset(obs)
    act = torch.zeros(n, dtype=torch.uint8, device="cuda")
    tiny.step(act, obs, rew, done)
    tiny.check()
    tiny.counts_map_sum(out)  # one block per env so far: the pool still holds
    exhausted = False
    for s in range(1, 20):
        for k, e in enumerate((1, 17, 40)):
            tiny.write_mem(e, 0xD35E, [(7 * s + 31 * k) % 248])
            tiny.write_mem(e, 0xD361, [(37 * s + 5 * k) % 250])
            tiny.write_mem(e, 0xD362, [(11 * s + 3 * k) % 250])
        try:
            tiny.step(act, obs, rew, done)
            tiny.check()
        except _capi.GbEnvError as err:
            assert "heat-map block pool" in str(err)
            exhausted = True
            break
    assert exhausted
    with pytest.raises(_capi.GbEnvError, match="heat-map block pool"):
        tiny.counts_map_sum(out)
