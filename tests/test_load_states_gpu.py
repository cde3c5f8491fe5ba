"""Batched load-states on the device (gbenv_load_states: k_load_check + k_load_states): rows written by gbenv_save_states
load into any envs exactly as gbenv_add_state_template + gbenv_load_template and the CPU oracle load the same bytes, for
any ids, with rejected rows leaving their envs untouched, across streams, composed with resets, and through
VecEnvironment.load_states."""
import ctypes as C

import numpy as np
import pytest

from helpers import GOLDEN
from pokegym_b200 import _capi
from pokegym_b200.state_file import diff_states, field_offsets

pytestmark = pytest.mark.gpu

S = _capi.STATE_BYTES
E_ARG, E_STATE = -1, -2
F = field_offsets(9)
STAT = F["lcd_regs"][0] + 4
CLOCK_HIGH = F["lcd_clock"][0] + 2 + 4
CART_RAM = F["cart_ram"][0]


def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _mixed(h, n, offset=0):
    """env i starts from mixed reference state (i + offset) mod 40"""
    states = np.load(GOLDEN / "red_states_mixed.npz")["states"]
    for k in range(len(states)):
        ids = np.arange(k, n, len(states), dtype=np.int32)
        if ids.size:
            h.load_template(h.add_state_template(states[(k + offset) % len(states)].tobytes()), ids)


def _rows(h, n):
    """save_states of envs 0..n-1, on the host"""
    import torch

    if h.lib.prefix == "oracle_":
        out = np.zeros((n, S), np.uint8)
        h.save_states(out)
        return out
    out = torch.empty((n, S), dtype=torch.uint8, device="cuda")
    h.save_states(out)
    return out.cpu().numpy()


def _load(h, rows, ids=None):
    """load_states of host rows into h, returning the status"""
    import torch

    rows = np.array(rows)  # a copy: a slice of a row array is not 16-byte aligned
    if h.lib.prefix == "oracle_":
        status = np.full(len(rows), 99, np.int32)
        h.load_states(rows, None if ids is None else np.asarray(ids, np.int32), status)
        return status
    status = torch.full((len(rows),), 99, dtype=torch.int32, device="cuda")
    h.load_states(_dev(rows), None if ids is None else _dev(np.asarray(ids, np.int32)), status)
    return status.cpu().numpy()


def _extra(h, n):
    return np.array([(x.stat_mode, x.ly_window) for x in (h.core_extra(e) for e in range(n))])


def _first_diff(a, b, where):
    bad = [i for i in range(len(a)) if not np.array_equal(a[i], b[i])]
    if bad:
        raise AssertionError(f"{where}: {len(bad)} rows differ, first env {bad[0]}: {diff_states(a[bad[0]].tobytes(), b[bad[0]].tobytes())[:4]}")


def _same(a, b, n, where):
    _first_diff(_rows(a, n), _rows(b, n), where)
    assert np.array_equal(_extra(a, n), _extra(b, n)), f"{where}: STAT mode / ly_window"


def _step_all(hs, n, rng):
    act = rng.integers(0, 8, n).astype(np.uint8)
    for h in hs:
        h.run_action(act if h.lib.prefix == "oracle_" else _dev(act))


@pytest.mark.parametrize("n", [1, 31, 33, 4096])
def test_parity_with_templates_and_oracle(cuda_lib, oracle_lib, roms, n):
    """Rows of a source handle after 0, 1 and 50 steps, loaded with permuted ids into a handle that has its own history:
    the same as the oracle's load_states, and as one template per row on the GPU where 1,024 templates suffice; then 20
    identical steps keep them identical.  At 4,096 envs every row is a distinct state, which the template path cannot load."""
    rom = roms("pokelike")
    src = _capi.Handle(cuda_lib, n, rom, 0)
    _mixed(src, n)
    dst, ref = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    tmpl = _capi.Handle(cuda_lib, n, rom, 0) if 3 * n <= 1024 else None
    targets = [h for h in (dst, ref, tmpl) if h is not None]
    for h in targets:
        _mixed(h, n, offset=17)
        h.tick(7, True)
    rng = np.random.default_rng(n)
    done = 0
    for steps in (0, 1, 50):
        for _ in range(steps - done):
            _step_all([src], n, rng)
        done = steps
        rows = _rows(src, n)
        rows[:, CART_RAM : CART_RAM + 4] = np.arange(n, dtype=np.uint32).view(np.uint8).reshape(n, 4)  # every row distinct
        ids = rng.permutation(n).astype(np.int32)
        assert (_load(dst, rows, ids) == 0).all()
        assert (_load(ref, rows, ids) == 0).all()
        if tmpl is not None:
            for i in range(n):
                tmpl.load_template(tmpl.add_state_template(rows[i].tobytes()), [int(ids[i])])
            _same(dst, tmpl, n, f"{steps} steps: templates")
        _same(dst, ref, n, f"{steps} steps: oracle")
        inv = np.argsort(ids)
        got = _rows(dst, n)
        assert not (got != rows[inv])[:, np.arange(S) != STAT].any(), "a loaded row differs outside STAT"
    for t in range(20):
        _step_all(targets, n, rng)
        if t in (0, 19):
            _same(dst, ref, n, f"step {t} after the load: oracle")
            if tmpl is not None:
                _same(dst, tmpl, n, f"step {t} after the load: templates")


def test_identity_and_twin(cuda_lib, roms):
    import torch

    n = 77
    rom = roms("pokelike")
    a, b = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(cuda_lib, n, rom, 0)
    rng = np.random.default_rng(1)
    for h in (a, b):
        _mixed(h, n)
    for _ in range(5):
        _step_all([a, b], n, rng)
    rows = torch.empty((n, S), dtype=torch.uint8, device="cuda")
    a.save_states(rows)
    before = rows.cpu().numpy()
    a.load_states(rows)
    assert np.array_equal(_rows(a, n), before)
    _same(a, b, n, "after loading its own rows")
    for _ in range(20):
        _step_all([a, b], n, rng)
    _same(a, b, n, "20 steps after loading its own rows")


def _pair(cuda_lib, oracle_lib, roms, n):
    rom = roms("pokelike")
    src = _capi.Handle(cuda_lib, n, rom, 0)
    _mixed(src, n, offset=5)
    _step_all([src], n, np.random.default_rng(2))
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    for h in (gpu, cpu):
        _mixed(h, n)
    return _rows(src, n), gpu, cpu


def test_id_semantics(cuda_lib, oracle_lib, roms):
    n = 70
    rows, gpu, cpu = _pair(cuda_lib, oracle_lib, roms, n)
    cases = [np.arange(n)[::-1], np.arange(0, n, 3), np.array([7, 7, 0, 69, 7, 1] * 5), np.arange(9, 69),
             np.array([3, -1, 4, n, n, 5, 1 << 30, 6, -1, -(1 << 30)])]
    for k, ids in enumerate(cases):
        ids = ids.astype(np.int32)
        blob = rows[(np.arange(len(ids)) * 7 + k) % n]
        st_g, st_c = _load(gpu, blob, ids), _load(cpu, blob, ids)
        assert np.array_equal(st_g, st_c), k
        assert np.array_equal(st_g, np.where((ids >= 0) & (ids < n), 0, E_ARG)), k
        _same(gpu, cpu, n, f"case {k}")
    # NULL ids with n < n_envs: envs 0..39 only
    before = _rows(gpu, n)
    assert (_load(gpu, rows[10:50]) == 0).all()
    _load(cpu, rows[10:50])
    _same(gpu, cpu, n, "NULL ids")
    after = _rows(gpu, n)
    assert np.array_equal(after[40:], before[40:])
    assert not (after[:40] != rows[10:50])[:, np.arange(S) != STAT].any()
    # envs not listed stay untouched
    before = _rows(gpu, n)
    _load(gpu, rows[:3], [11, 12, 13])
    after = _rows(gpu, n)
    keep = np.setdiff1d(np.arange(n), [11, 12, 13])
    assert np.array_equal(after[keep], before[keep])


def _corrupt(rows):
    """(name, row) for each rule: version byte, cgb byte, high halves of clock and clock_target, a screen word"""
    so = F["screen"][0]
    out = []
    for name, o, v in [("version", 0, 7), ("cgb", 4, 1), ("clock high", CLOCK_HIGH, 1), ("target high", CLOCK_HIGH + 8 + 3, 0x80),
                       ("screen word 0", so, 0x02), ("last screen word", so + F["screen"][1] - 3, 0x42)]:
        r = rows[len(out) % len(rows)].copy()
        r[o] = v
        out.append((name, r))
    return out


def test_rejected_rows_leave_their_envs_untouched(cuda_lib, oracle_lib, roms):
    n = 40
    rows, gpu, cpu = _pair(cuda_lib, oracle_lib, roms, n)
    bad = _corrupt(rows)
    before = _rows(gpu, n)
    ids = np.arange(len(bad), dtype=np.int32) * 3 + 1
    # valid rows in between still load
    blob = np.concatenate([np.stack([r for _, r in bad]), rows[20:24]])
    all_ids = np.concatenate([ids, [30, 31, 32, 33]]).astype(np.int32)
    for h in (gpu, cpu):
        st = _load(h, blob, all_ids)
        assert st.tolist() == [E_STATE] * len(bad) + [0] * 4, st
    after = _rows(gpu, n)
    assert np.array_equal(after[ids], before[ids]), [name for (name, _), e in zip(bad, ids) if not np.array_equal(after[e], before[e])]
    assert not (after[30:34] != rows[20:24])[:, np.arange(S) != STAT].any()
    _same(gpu, cpu, n, "after rejected rows")
    # a later invalid duplicate does not override an earlier valid entry; a later valid one does
    blob = np.stack([rows[5], bad[1][1], rows[6], rows[7], bad[4][1]])
    ids = np.array([2, 2, 3, 3, 3], np.int32)
    for h in (gpu, cpu):
        assert _load(h, blob, ids).tolist() == [0, E_STATE, 0, 0, E_STATE]
    after = _rows(gpu, n)
    assert not (after[[2, 3]] != rows[[5, 7]])[:, np.arange(S) != STAT].any()
    _same(gpu, cpu, n, "duplicates")


def test_argument_errors(cuda_lib, roms):
    import torch

    n = 40
    h = _capi.Handle(cuda_lib, n, roms("pokelike"), 0)
    _mixed(h, n)
    before = _rows(h, n)
    buf = torch.zeros((n + 2) * S + 16, dtype=torch.uint8, device="cuda")
    buf[: n * S].copy_(torch.from_numpy(before.reshape(-1)))
    ids = _dev(np.arange(4, dtype=np.int32))
    status = torch.zeros(8, dtype=torch.int32, device="cuda")
    p, hp, lib = buf.data_ptr(), h._h, cuda_lib
    sp, ip = status.data_ptr(), ids.data_ptr()
    assert lib.load_states(None, None, 4, C.c_void_p(p), None, None) == E_ARG  # NULL handle
    assert lib.load_states(hp, None, 4, None, None, None) == E_ARG  # NULL rows, n > 0
    for mis in (1, 2, 8):
        assert lib.load_states(hp, None, 4, C.c_void_p(p + mis), None, None) == E_ARG  # rows not 16-byte aligned
    assert lib.load_states(hp, C.c_void_p(ip + 2), 1, C.c_void_p(p), None, None) == E_ARG  # ids not 4-byte aligned
    assert lib.load_states(hp, None, 4, C.c_void_p(p), C.c_void_p(sp + 1), None) == E_ARG  # status not 4-byte aligned
    assert lib.load_states(hp, None, -1, C.c_void_p(p), None, None) == E_ARG  # n < 0
    assert lib.load_states(hp, None, n + 1, C.c_void_p(p), None, None) == E_ARG  # NULL ids with n > n_envs
    assert lib.load_states(hp, C.c_void_p(ip), 0, None, None, None) == 0  # n == 0: no-op, even with no rows
    assert lib.load_states(hp, None, 0, None, None, None) == 0
    h.sync()
    assert np.array_equal(_rows(h, n), before)  # nothing was loaded by the refused calls
    assert lib.load_states(hp, C.c_void_p(ip), 4, C.c_void_p(p), C.c_void_p(sp), None) == 0
    h.sync()
    assert status[:4].tolist() == [0, 0, 0, 0]
    with pytest.raises(ValueError):
        h.load_states(buf[1 : 1 + 4 * S], ids)  # misaligned rows are refused before the pointer crosses the ABI
    with pytest.raises(ValueError):
        h.load_states(buf[: 3 * S], ids)  # fewer rows than ids
    with pytest.raises(ValueError):
        h.load_states(buf[: 4 * S], ids, status)  # status of the wrong length
    with pytest.raises(ValueError):
        h.load_states(buf[: 4 * S], ids, torch.zeros(4, dtype=torch.int64, device="cuda"))


def test_stream_order(cuda_lib, roms):
    import torch

    n = 96
    rom = roms("pokelike")
    a, b = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(cuda_lib, n, rom, 0)
    for h in (a, b):
        _mixed(h, n)
    src = _capi.Handle(cuda_lib, n, rom, 0)
    _mixed(src, n, offset=9)
    rows = torch.empty((n, S), dtype=torch.uint8, device="cuda")
    src.save_states(rows)
    ids = _dev(np.arange(n, dtype=np.int32)[::-1].copy())
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    g = torch.Generator(device="cuda").manual_seed(11)
    acts = [torch.randint(0, 8, (n,), generator=g, device="cuda", dtype=torch.uint8) for _ in range(3)]
    torch.cuda.synchronize()
    for t in range(3):
        a.run_action(acts[t], stream=s1.cuda_stream)
        a.load_states(rows, ids if t % 2 else None, stream=s2.cuda_stream)  # ordered after the step on the other stream
        a.run_action(acts[t], stream=s1.cuda_stream)  # ... and before this one
        b.run_action(acts[t], stream=s1.cuda_stream)
        b.load_states(rows, ids if t % 2 else None, stream=s1.cuda_stream)
        b.run_action(acts[t], stream=s1.cuda_stream)
        torch.cuda.synchronize()
        _same(a, b, n, f"round {t}")


def _initial_templates(hs, n):
    states = np.load(GOLDEN / "red_states_mixed.npz")["states"]
    for h in hs:
        for k in range(8):
            h.set_initial_template(h.add_state_template(states[k].tobytes()), np.arange(k, n, 8, dtype=np.int32))


def _buffers(n):
    import torch

    return ((torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda"),
             torch.zeros(n, dtype=torch.uint8, device="cuda")), (np.zeros((n, _capi.OBS_BYTES), np.uint8), np.zeros(n), np.zeros(n, np.uint8)))


def test_reset_composition(cuda_lib, oracle_lib, roms):
    """After the first reset: load_states + reset_dev(mask) equals the oracle's load_template + reset(mask), in observations,
    rewards, dones and info rows over the following steps."""
    import torch

    n = 64
    rom = roms("pokelike")
    src = _capi.Handle(cuda_lib, n, rom, 0)
    _mixed(src, n, offset=21)
    _step_all([src], n, np.random.default_rng(4))
    rows = _rows(src, n)
    gpu, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    _initial_templates([gpu, cpu], n)
    (og, rg, dg), (oc, rc, dc) = _buffers(n)
    gpu.reset_dev(og, None, max_episode_steps=40)
    cpu.reset(oc, None, max_episode_steps=40)
    rng = np.random.default_rng(6)

    def step(t):
        act = rng.integers(0, 8, n).astype(np.uint8)
        gpu.step(_dev(act), og, rg, dg)
        cpu.step(act, oc, rc, dc)
        assert np.array_equal(og.cpu().numpy(), oc), f"obs, step {t}"
        assert np.array_equal(rg.cpu().numpy(), rc), f"reward, step {t}"
        assert np.array_equal(dg.cpu().numpy(), dc), f"done, step {t}"

    for t in range(3):
        step(t)
    ids = rng.permutation(n).astype(np.int32)
    _load(gpu, rows, ids)
    for i, e in enumerate(ids):
        cpu.load_template(cpu.add_state_template(rows[i].tobytes()), [int(e)])
    mask = np.zeros(n, np.uint8)
    mask[::3] = 1
    gpu.reset_dev(og, _dev(mask), max_episode_steps=40)
    cpu.reset(oc, mask, max_episode_steps=40)
    assert np.array_equal(og.cpu().numpy()[mask == 1], oc[mask == 1])
    _same(gpu, cpu, n, "after load_states + reset")
    for t in range(3, 30):
        step(t)
    ig = torch.zeros((n, _capi.INFO_SCALARS), dtype=torch.float64, device="cuda")
    ic = np.zeros((n, _capi.INFO_SCALARS))
    gpu.get_info(ig)
    cpu.get_info(ic)
    gpu.sync()
    assert np.array_equal(ig.cpu().numpy(), ic)


def test_first_reset_loads_the_initial_template(cuda_lib, oracle_lib, roms):
    """An env whose first reset is still ahead loads its initial template on that reset, whatever load_states put there."""
    n = 40
    rom = roms("pokelike")
    src = _capi.Handle(cuda_lib, n, rom, 0)
    _mixed(src, n, offset=13)
    rows = _rows(src, n)
    gpu, twin, cpu = _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(cuda_lib, n, rom, 0), _capi.Handle(oracle_lib, n, rom)
    _initial_templates([gpu, twin, cpu], n)
    assert (_load(gpu, rows[:20], np.arange(0, 40, 2)) == 0).all()
    _load(cpu, rows[:20], np.arange(0, 40, 2))
    (og, _, _), (oc, _, _) = _buffers(n)
    (ot, _, _), _ = _buffers(n)
    gpu.reset_dev(og, None)
    twin.reset_dev(ot, None)
    cpu.reset(oc, None)
    import torch

    assert torch.equal(og, ot) and np.array_equal(og.cpu().numpy(), oc)
    _same(gpu, twin, n, "first reset after load_states vs no load")
    _same(gpu, cpu, n, "first reset after load_states: oracle")


@pytest.mark.parametrize("obs_format", ["reference", "packed"])
def test_vec_environment_load_states(cuda_lib, roms, obs_format):
    import torch

    from pokegym_b200 import VecEnvironment

    n = 48
    blobs = [b.tobytes() for b in np.load(GOLDEN / "red_states_mixed.npz")["states"][:8]]
    vecs = [VecEnvironment(n, roms("pokelike"), blobs, max_episode_steps=30, auto_reset=True, obs_format=obs_format) for _ in range(2)]
    for v in vecs:
        v.reset()
    g = torch.Generator(device="cuda").manual_seed(3)
    for _ in range(4):
        act = torch.randint(0, 8, (n,), generator=g, device="cuda", dtype=torch.uint8)
        for v in vecs:
            v.step(act)
    rows = vecs[0].save_states()
    perm = np.random.default_rng(0).permutation(n)
    # device rows
    st = vecs[1].load_states(rows[torch.from_numpy(perm).cuda()], list(range(n)))
    assert st.dtype == torch.int32 and st.shape == (n,) and (st == 0).all()
    got = vecs[1].save_states().cpu().numpy()
    want = rows.cpu().numpy()[perm]
    assert not (got != want)[:, np.arange(S) != STAT].any()
    # host rows, into some envs
    host = want[:5][::-1].copy()
    st = vecs[1].load_states(host, [40, 41, 42, 43, 44])
    assert (st == 0).all()
    assert not (vecs[1].save_states([40, 41, 42, 43, 44]).cpu().numpy() != host)[:, np.arange(S) != STAT].any()
    # misaligned device rows (a slice that starts 142,610 B into a buffer) and a corrupt row
    big = torch.empty((n + 1, S), dtype=torch.uint8, device="cuda")
    big[1:].copy_(rows)
    big[1 + 7, 0] = 7
    st = vecs[0].load_states(big[1:])
    assert st[7].item() == E_STATE and (st[torch.arange(n, device="cuda") != 7] == 0).all()
    assert torch.equal(vecs[0].save_states(), rows)
    # the broadcast idiom
    one = rows[3]
    st = vecs[0].load_states(one.expand(4, -1).contiguous(), [0, 1, 2, 3])
    assert (st == 0).all()
    assert not (vecs[0].save_states([0, 1, 2, 3]).cpu().numpy() != rows[3].cpu().numpy())[:, np.arange(S) != STAT].any()
    # wrong shapes
    for bad_rows, ids in ((rows[:, :-1], None), (rows[0], None), (rows[:4], [1, 2]), (torch.zeros((n + 1, S), dtype=torch.uint8), None),
                          (rows.to(torch.int16), None)):
        with pytest.raises(ValueError):
            vecs[0].load_states(bad_rows, ids)
    with pytest.raises(ValueError):
        vecs[0].load_states(rows[:2], [0, n])
    # stepping goes on in the chosen observation format
    act = torch.randint(0, 8, (n,), generator=g, device="cuda", dtype=torch.uint8)
    obs = vecs[0].step(act)[0]
    assert obs.shape[0] == n and obs.dtype == torch.uint8
    torch.cuda.synchronize()
