"""Episode-end reductions on the CPU oracle: the heat-map sum (gbenv_counts_map_sum) and the masked info sum
(gbenv_reduce_info_masked), and the exploration-map sum all-reduced over two gloo ranks."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from pokegym_b200 import _capi

MAP_SHAPE = (_capi.COUNTS_H, _capi.COUNTS_W)


def _walk(h, n, steps, seed, mask_reset_at=None, max_episode_steps=20480):
    """n envs, `steps` random actions; envs 1 and n - 2 are teleported to a new map every step, so their maps hold many
    cells and the -1 marks map transitions leave.  Optionally a masked reset (odd envs) before step `mask_reset_at`."""
    h.tick(30, True)
    obs, rew, done = np.zeros((n, _capi.OBS_BYTES), np.uint8), np.zeros(n), np.zeros(n, np.uint8)
    h.reset(obs, max_episode_steps=max_episode_steps)
    rng = np.random.default_rng(seed)
    for s in range(steps):
        if s == mask_reset_at:
            h.reset(obs, mask=(np.arange(n) % 2).astype(np.uint8), max_episode_steps=max_episode_steps)
        for k, e in enumerate((1, n - 2)):
            h.write_mem(e, 0xD35E, [(7 * s + 31 * k) % 248])
            h.write_mem(e, 0xD361, [(37 * s + 5 * k) % 250])
            h.write_mem(e, 0xD362, [(11 * s + 3 * k) % 250])
        h.step(rng.integers(0, 8, n).astype(np.uint8), obs, rew, done)
    return done


def _per_env_sum(h, envs):
    total = np.zeros(MAP_SHAPE, np.int64)
    for e in envs:
        total += h.counts_map(e)
    return total


def test_oracle_map_sum_equals_per_env_maps(oracle_lib, roms):
    n = 12
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    _walk(h, n, 24, seed=1)
    out = np.full(MAP_SHAPE, 7, np.int64)  # overwritten, not accumulated into
    h.counts_map_sum(out)
    assert np.array_equal(out, _per_env_sum(h, range(n)))
    assert (out < 0).any() and (out > 0).sum() > 20  # the walkers left -1 marks and many visited cells
    rng = np.random.default_rng(4)
    mask = (rng.random(n) < 0.5).astype(np.uint8)
    mask[[1, 2]] = 1, 0
    h.counts_map_sum(out, mask)
    assert np.array_equal(out, _per_env_sum(h, np.nonzero(mask)[0]))
    h.counts_map_sum(out, np.zeros(n, np.uint8))
    assert not out.any()


def test_oracle_map_sum_keeps_accumulating_across_a_masked_reset(oracle_lib, roms):
    """The heat map lives as long as the env: a reset does not clear it, so the sum only grows for envs that keep walking."""
    n = 8
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    _walk(h, n, 10, seed=2)
    before = np.zeros(MAP_SHAPE, np.int64)
    h.counts_map_sum(before)
    obs = np.zeros((n, _capi.OBS_BYTES), np.uint8)
    h.reset(obs, mask=(np.arange(n) % 2).astype(np.uint8))
    after_reset = np.zeros(MAP_SHAPE, np.int64)
    h.counts_map_sum(after_reset)
    assert np.array_equal(after_reset, before)
    rew, done = np.zeros(n), np.zeros(n, np.uint8)
    for _ in range(3):
        h.step(np.zeros(n, np.uint8), obs, rew, done)
    later = np.zeros(MAP_SHAPE, np.int64)
    h.counts_map_sum(later)
    assert np.array_equal(later, _per_env_sum(h, range(n)))
    assert later.sum() > before.sum()


def test_oracle_masked_info_sum(oracle_lib, roms):
    n = 10
    h = _capi.Handle(oracle_lib, n, roms("pokelike"))
    _walk(h, n, 8, seed=3)
    full, masked_all = np.zeros(_capi.INFO_SCALARS), np.zeros(_capi.INFO_SCALARS)
    h.reduce_info(full)
    h.reduce_info_masked(masked_all)
    assert np.array_equal(full, masked_all)
    rows = np.zeros((n, _capi.INFO_SCALARS))
    h.get_info(rows)
    mask = np.zeros(n, np.uint8)
    mask[[0, 3, 4, 9]] = 1
    part = np.zeros(_capi.INFO_SCALARS)
    h.reduce_info_masked(part, mask)
    assert part[0] == 4  # slot 0 counts the masked envs that have stepped
    assert np.allclose(part, rows[mask.astype(bool)].sum(axis=0), rtol=1e-12, atol=0)
    h.reduce_info_masked(part, np.zeros(n, np.uint8))
    assert not part.any()
    fresh = _capi.Handle(oracle_lib, 3, roms("pokelike"))  # no env has stepped: slot 0 is 0
    fresh.reduce_info_masked(part, np.ones(3, np.uint8))
    assert part[0] == 0


def _worker(rank, world, port, n_total, steps, lib_path, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from pokegym_b200.dist import all_reduce_info, shard_range
    from pokegym_b200.tools import synth_rom

    lo, hi = shard_range(n_total, rank, world)
    h = _capi.Handle(_capi.GbEnvLib(lib_path, "oracle_"), hi - lo, synth_rom.build_pokelike_rom())
    h.tick(30, True)
    obs, rew, done = np.zeros((hi - lo, _capi.OBS_BYTES), np.uint8), np.zeros(hi - lo), np.zeros(hi - lo, np.uint8)
    h.reset(obs)
    actions = np.random.default_rng(0).integers(0, 8, (steps, n_total)).astype(np.uint8)
    for s in range(steps):
        h.step(np.ascontiguousarray(actions[s, lo:hi]), obs, rew, done)
    local = np.zeros(MAP_SHAPE, np.int64)
    h.counts_map_sum(local)
    total = torch.from_numpy(local)
    all_reduce_info(total)
    q.put((rank, total.numpy().copy()))
    dist.destroy_process_group()


def test_two_rank_map_sum_matches_single_process(built):
    n_total, steps, world = 6, 6, 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_total, steps, str(built["oracle"]), q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=180) for _ in range(world)), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    from pokegym_b200.tools import synth_rom

    h = _capi.Handle(_capi.GbEnvLib(built["oracle"], "oracle_"), n_total, synth_rom.build_pokelike_rom())
    h.tick(30, True)
    obs, rew, done = np.zeros((n_total, _capi.OBS_BYTES), np.uint8), np.zeros(n_total), np.zeros(n_total, np.uint8)
    h.reset(obs)
    actions = np.random.default_rng(0).integers(0, 8, (steps, n_total)).astype(np.uint8)
    for s in range(steps):
        h.step(actions[s], obs, rew, done)
    ref = np.zeros(MAP_SHAPE, np.int64)
    h.counts_map_sum(ref)
    assert ref.sum() > 0
    assert res[0][1].dtype == np.int64
    assert np.array_equal(res[0][1], ref) and np.array_equal(res[1][1], ref)
