"""Packed observations on the device (gbenv_step_packed / gbenv_reset_packed / k_obs_pack, gbenv_unpack_obs / k_obs_unpack):
twin runs of two identical handles, one on the reference calls and one on the packed calls, agree bit for bit on every
output; the shades are the framebuffer's; VecEnvironment, PufferVecAdaptor and EnvGroups in packed mode deliver what the
reference-format objects deliver; the error paths."""
import numpy as np
import pytest

from pokegym_b200 import _capi

from test_obs_packed_cpu import E_ARG, SENTINEL

pytestmark = pytest.mark.gpu

PB, OB = _capi.OBS_PACKED_BYTES, _capi.OBS_BYTES


def _mixed_blobs():
    from helpers import GOLDEN

    return [b.tobytes() for b in np.load(GOLDEN / "red_states_mixed.npz")["states"]]


def _start(h, n, blobs):
    if blobs is None:
        h.tick(60, True)
        return
    for k, blob in enumerate(blobs):
        ids = np.arange(k, n, len(blobs), dtype=np.int32)
        if ids.size:
            h.set_initial_template(h.add_state_template(blob), ids)


class Twin:
    """Handle `a` on step_masked / reset_dev, handle `b` on step_packed / reset_packed, built and driven identically."""

    def __init__(self, cuda_lib, rom, n, blobs=None, lanes=None, mes=50):
        import torch

        self.torch, self.n, self.mes = torch, n, mes
        self.a, self.b = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(cuda_lib, n, rom, 0)
        for h in (self.a, self.b):
            if lanes:
                h.set_lanes_per_warp(lanes)
            _start(h, n, blobs)
        z = lambda *shape, dt=torch.uint8: torch.zeros(shape, dtype=dt, device="cuda")  # noqa: E731
        self.obs, self.packed, self.out = z(n, OB), z(n, PB), z(n, OB)
        self.ra, self.rb, self.da, self.db = z(n, dt=torch.float64), z(n, dt=torch.float64), z(n), z(n)
        self.ia, self.ib = z(n, _capi.INFO_SCALARS, dt=torch.float64), z(n, _capi.INFO_SCALARS, dt=torch.float64)
        self.resets = 0

    def compare(self, rows, where):
        torch = self.torch
        self.b.unpack_obs(self.packed, self.out)
        rows = torch.as_tensor(rows, device="cuda")
        assert torch.equal(self.out[rows], self.obs[rows]), f"{where}: unpacked observation differs from the reference one"

    def reset(self, mask=None, where="reset"):
        self.a.reset_dev(self.obs, mask, max_episode_steps=self.mes)
        self.b.reset_packed(self.packed, mask, max_episode_steps=self.mes)
        rows = np.arange(self.n) if mask is None else np.nonzero(mask.cpu().numpy())[0]
        self.compare(rows, where)
        self.resets += 1

    def step(self, act, skip, where):
        torch = self.torch
        if skip is not None:  # PufferLib's skip path: the rows of envs that sit out come back untouched
            self.obs[skip.bool()] = SENTINEL
            self.packed[skip.bool()] = SENTINEL
        self.a.step_masked(act, skip, self.obs, self.ra, self.da)
        self.b.step_packed(act, skip, self.packed, self.rb, self.db)
        assert torch.equal(self.ra, self.rb), f"{where}: reward differs"
        assert torch.equal(self.da, self.db), f"{where}: done differs"
        self.a.get_info(self.ia)
        self.b.get_info(self.ib)
        assert torch.equal(self.ia, self.ib), f"{where}: info rows differ"
        if skip is None:
            self.compare(np.arange(self.n), where)
        else:
            s = skip.cpu().numpy()
            self.compare(np.nonzero(s == 0)[0], where)
            assert bool((self.packed[skip.bool()] == SENTINEL).all()), f"{where}: a skipped env's packed row was written"
        if bool(self.da.any()):  # auto-reset on done, masked on the device
            self.reset(self.da.clone(), f"{where}: auto-reset")

    def run(self, steps, seed):
        torch = self.torch
        gen = torch.Generator(device="cuda").manual_seed(seed)
        for s in range(steps):
            act = torch.randint(0, 8, (self.n,), generator=gen, device="cuda", dtype=torch.uint8)
            skip = (torch.rand(self.n, generator=gen, device="cuda") < 0.3).to(torch.uint8) if s % 3 == 2 else None
            self.step(act, skip, f"step {s}")

    def same_states(self, sample):
        for e in sample:
            assert self.a.save_state(int(e)) == self.b.save_state(int(e)), f"env {e}: emulator state differs"
        self.a.check()
        self.b.check()


@pytest.mark.parametrize("n,lanes,mixed", [(1, 1, False), (33, 16, True), (72, 32, True), (72, 1, False), (4096, None, True)])
def test_twin_run_packed_equals_reference(cuda_lib, roms, n, lanes, mixed):
    """200 steps with skips on every third step and auto-resets on done: after every step and reset the unpacked rows equal
    the reference rows; rewards, dones and info rows are bit-identical; emulator states at the end too."""
    t = Twin(cuda_lib, roms("pokelike"), n, _mixed_blobs() if mixed else None, lanes, mes=50)
    t.reset()
    t.run(200, seed=n)
    assert t.resets > 1  # some episode ended and was reset
    t.same_states(sorted({0, n // 2, n - 1}))


def test_twin_run_replicated_full_batch(cuda_lib, roms):
    """32,768 envs, env i from reference save-state i mod 40: the packed writer over many tiles, maps and positions."""
    n = 32768
    t = Twin(cuda_lib, roms("pokelike"), n, _mixed_blobs(), mes=6)
    t.reset()
    t.run(14, seed=7)
    assert t.resets > 1
    t.same_states([0, 31, 32, 12345, n - 1])


def test_packed_shades_are_the_framebuffer_shades(cuda_lib, roms):
    """Shade of obs pixel (i, j) == shade of framebuffer pixel (2j, 2i) of capture_frames on the same state."""
    import torch

    n = 64
    h = _capi.Handle(cuda_lib, n, roms("pokelike"), 0)
    h.tick(60, True)
    packed = torch.zeros((n, PB), dtype=torch.uint8, device="cuda")
    rew, done = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.uint8, device="cuda")
    h.reset_packed(packed)
    gen = torch.Generator(device="cuda").manual_seed(3)
    distinct = set()
    for s in range(4):
        h.step_packed(torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8), None, packed, rew, done)
        frames = torch.empty((n, _capi.FRAME_WORDS), dtype=torch.int32, device="cuda")
        h.capture_frames(frames)
        fw = frames.cpu().numpy().view(np.uint32).reshape(n, 144, 10)
        pw = packed.cpu().numpy().view(np.uint32).reshape(n, 72, 8)
        i, j = np.meshgrid(np.arange(72), np.arange(80), indexing="ij")
        fb_shade = (fw[:, 2 * i, (2 * j) // 16] >> (2 * ((2 * j) & 15)).astype(np.uint32)) & 3
        obs_shade = (pw[:, i, j // 16] >> (2 * (j & 15)).astype(np.uint32)) & 3
        assert np.array_equal(obs_shade, fb_shade), f"step {s}"
        assert (pw[:, :, 7] >> 16 == 0).all()  # bits of pixels j >= 80 are 0
        distinct.update(r.tobytes() for r in pw)
    assert len(distinct) > 1


def test_vec_environment_packed_rollout_matches_reference(cuda_lib, roms):
    import torch

    from pokegym_b200.vec_env import VecEnvironment

    n, T, steps = 48, 4, 30
    rom = roms("pokelike")
    roll_r = torch.zeros((T, n, 72, 80, 4), dtype=torch.uint8, device="cuda")
    roll_p = torch.zeros((T, n, PB), dtype=torch.uint8, device="cuda")
    ref = VecEnvironment(n, rom, rollout=roll_r, auto_reset=True, max_episode_steps=10)
    pk = VecEnvironment(n, rom, rollout=roll_p, auto_reset=True, max_episode_steps=10, obs_format="packed")
    assert pk.observation_space.shape == (PB,) and ref.observation_space.shape == (72, 80, 4)
    o_r, _ = ref.reset()
    o_p, _ = pk.reset()
    assert o_p.shape == (n, PB) and o_p.data_ptr() == roll_p[0].data_ptr()
    assert torch.equal(pk.unpack_obs(o_p), o_r)
    gen = torch.Generator(device="cuda").manual_seed(11)
    ended = 0
    for s in range(steps):
        act = torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8)
        o_r, r_r, d_r, _, _ = ref.step(act)
        o_p, r_p, d_p, _, _ = pk.step(act)
        assert o_p.data_ptr() == roll_p[(s + 1) % T].data_ptr()
        assert torch.equal(pk.unpack_obs(o_p), o_r), f"step {s}"
        assert torch.equal(r_p, r_r) and torch.equal(d_p, d_r), f"step {s}"
        ended += int(d_r.sum())
    assert ended > 0  # auto_reset rows were compared
    full = pk.unpack_obs(roll_p)  # the whole ring, any leading dims
    assert full.shape == (T, n, 72, 80, 4) and torch.equal(full, roll_r)
    idx = torch.tensor([3, 0, 7, 7, 40], device="cuda")
    mb = roll_p.view(T * n, PB)[idx]  # a minibatch gathered from the ring
    out = torch.empty((len(idx), 72, 80, 4), dtype=torch.uint8, device="cuda")
    assert pk.unpack_obs(mb, out=out) is out and torch.equal(out, roll_r.view(T * n, 72, 80, 4)[idx])
    assert torch.equal(pk.compact_view(out), out[..., 2:])
    assert pk.unpack_obs(roll_p[:, :0]).shape == (T, 0, 72, 80, 4)
    with pytest.raises(ValueError):
        pk.unpack_obs(roll_p[..., :100])
    with pytest.raises(ValueError):
        VecEnvironment(n, rom, obs_format="compact")
    with pytest.raises(ValueError):  # a reference-sized rollout for a packed vec
        VecEnvironment(n, rom, rollout=roll_r, obs_format="packed").reset()


def test_puffer_adaptor_over_packed_vec_matches_reference(cuda_lib, roms):
    import torch

    from pokegym_b200.puffer import PufferVecAdaptor
    from pokegym_b200.vec_env import VecEnvironment

    n, steps = 40, 36
    rom = roms("pokelike")
    vr = VecEnvironment(n, rom, max_episode_steps=8)
    vp = VecEnvironment(n, rom, max_episode_steps=8, obs_format="packed")
    ar, ap = PufferVecAdaptor(vr), PufferVecAdaptor(vp)
    ar.async_reset()
    ap.async_reset()
    gen = torch.Generator(device="cuda").manual_seed(5)
    ended = 0
    for s in range(steps):
        fr, rr, dr, _, ir, _, _ = ar.recv()
        fp, rp, dp, _, ip, _, _ = ap.recv()
        assert fp.shape == (n, PB) and fr.shape == (n, OB)
        assert torch.equal(vp.unpack_obs(fp).view(n, OB), fr), f"step {s}"
        assert torch.equal(rp, rr) and torch.equal(dp, dr) and ip == ir, f"step {s}"
        ended += len(ir)
        act = torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8)
        ar.send(act)
        ap.send(act)
    assert ended > 0  # resets on the call after done, with those envs skipped, were compared


def test_env_groups_packed_matches_one_handle(cuda_lib, roms):
    import torch

    from pokegym_b200.groups import EnvGroups

    n, steps = 256, 12
    rom = roms("pokelike")
    groups = EnvGroups(cuda_lib, n, rom, n_groups=2, obs_format="packed")
    one = _capi.Handle(cuda_lib, n, rom, 0)
    groups.for_each(lambda h, g, st: h.tick(60, True, stream=st))
    one.tick(60, True)
    z = lambda *shape, dt=torch.uint8: torch.zeros(shape, dtype=dt, device="cuda")  # noqa: E731
    pg, po, rg, ro, dg, do = z(n, PB), z(n, PB), z(n, dt=torch.float64), z(n, dt=torch.float64), z(n), z(n)
    groups.reset(pg, max_episode_steps=5)
    one.reset_packed(po, max_episode_steps=5)
    assert torch.equal(pg, po)
    gen = torch.Generator(device="cuda").manual_seed(9)
    for s in range(steps):
        act = torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8)
        groups.step(act, pg, rg, dg, join=True)
        one.step_packed(act, None, po, ro, do)
        assert torch.equal(pg, po) and torch.equal(rg, ro) and torch.equal(dg, do), f"step {s}"
        if bool(do.any()):
            mask = do.clone()
            groups.reset(pg, mask=mask, max_episode_steps=5)
            one.reset_packed(po, mask, max_episode_steps=5)
            assert torch.equal(pg, po), f"reset after step {s}"
    groups.close()


def test_cuda_packed_argument_errors(cuda_lib, roms):
    import torch

    n = 4
    h = _capi.Handle(cuda_lib, n, roms("pokelike"), 0)
    lib, hh, vp = h.lib, h._h, _capi._ptr
    z = lambda k, dt=torch.uint8: torch.zeros(k, dtype=dt, device="cuda")  # noqa: E731
    act, rew, done, packed, out = z(n), z(n, torch.float64), z(n), z(n * PB + 16), z(n * OB + 16)
    p, bad_p, o, bad_o = vp(packed), vp(packed.data_ptr() + 4), vp(out), vp(out.data_ptr() + 8)
    for args in ((None, None, p, vp(rew), vp(done)), (vp(act), None, None, vp(rew), vp(done)), (vp(act), None, p, None, vp(done)),
                 (vp(act), None, p, vp(rew), None), (vp(act), None, bad_p, vp(rew), vp(done))):
        assert lib.step_packed(hh, *args, None) == E_ARG
    assert lib.step_packed(None, vp(act), None, p, vp(rew), vp(done), None) == E_ARG
    assert lib.reset_packed(hh, None, 100, 4.0, None, None) == E_ARG
    assert lib.reset_packed(hh, None, 100, 4.0, bad_p, None) == E_ARG
    assert lib.reset_packed(None, None, 100, 4.0, p, None) == E_ARG
    for args in ((p, -1, o), (None, 1, o), (p, 1, None), (bad_p, 1, o), (p, 1, bad_o)):
        assert lib.unpack_obs(hh, *args, None) == E_ARG
    assert lib.unpack_obs(None, p, 1, o, None) == E_ARG
    out.fill_(SENTINEL)
    assert lib.unpack_obs(hh, None, 0, None, None) == 0
    assert lib.unpack_obs(hh, p, 0, o, None) == 0
    torch.cuda.synchronize()
    assert bool((out == SENTINEL).all())
    with pytest.raises(ValueError):
        h.step_packed(act, None, packed[1:1 + n * PB], rew, done)  # misaligned
    with pytest.raises(ValueError):
        h.unpack_obs(packed[:n * PB].view(n, PB), out[:(n - 1) * OB])
    h.check()
