"""Shared helpers for the parity tests."""
import hashlib
import json
import lzma
import zlib
from pathlib import Path

import numpy as np

from pokegym_b200 import _capi
from pokegym_b200.info import build_info
from pokegym_b200.state_file import field_offsets, parse_state, serialize_state

GOLDEN = Path(__file__).resolve().parent / "golden"
SHADE_WORDS = np.array([0xFFFFFF01, 0x99999900, 0x55555500, 0x00000000], dtype="<u4")


def info_fingerprint(info):
    """The reference's info dict (or build_info's) reduced to plain JSON-able data: numbers as floats, the exploration
    map as (sum, CRC32 of its int64 image), the reference's stray `set` under stats["maps_explored"] as its length."""
    if isinstance(info, dict):
        return {str(k): info_fingerprint(v) for k, v in info.items()}
    if isinstance(info, (set, frozenset)):
        return float(len(info))
    if isinstance(info, np.ndarray) and info.ndim:
        a = np.ascontiguousarray(info.astype(np.int64))
        return {"sum": float(a.sum()), "crc32": int(zlib.crc32(a.tobytes()))}
    if isinstance(info, (list, tuple)):
        return [info_fingerprint(v) for v in info]
    return float(info)


def replay_wrapper_golden(handle, gold, xp=None, to_dev=lambda a: a, to_host=lambda a: a):
    """Replays a ref_wrapper_*.npz recording through `handle` (oracle or CUDA) and checks every step."""
    n = 1
    start = gold["start_state"].tobytes()
    tid = handle.add_state_template(start)
    handle.set_initial_template(tid)
    obs = to_dev(np.zeros((n, _capi.OBS_BYTES), dtype=np.uint8))
    rew = to_dev(np.zeros(n, dtype=np.float64))
    done = to_dev(np.zeros(n, dtype=np.uint8))
    mes = int(gold["max_episode_steps"])
    reset_at = set(int(x) for x in gold["reset_at"])
    handle.reset(obs, max_episode_steps=mes)
    assert zlib.crc32(to_host(obs).tobytes()) == int(gold["reset_obs_crc"][0]), "reset observation differs from the reference"
    infos = {int(i): json.loads(str(t)) for i, t in zip(gold["info_steps"], gold["info_json"])} if "info_steps" in gold else {}
    info_row = to_dev(np.zeros((n, _capi.INFO_SCALARS), dtype=np.float64))
    k = 1
    for i, a in enumerate(gold["actions"]):
        if i in reset_at:
            handle.reset(obs, max_episode_steps=mes)
            assert zlib.crc32(to_host(obs).tobytes()) == int(gold["reset_obs_crc"][k]), f"observation of reset #{k + 1} differs"
            k += 1
        handle.step(to_dev(np.array([a], dtype=np.uint8)), obs, rew, done)
        r, d, o = float(to_host(rew)[0]), int(to_host(done)[0]), to_host(obs)
        assert r == float(gold["rewards"][i]), f"step {i}: reward {r!r} != reference {float(gold['rewards'][i])!r}"
        assert d == int(gold["dones"][i]), f"step {i}: done differs"
        assert zlib.crc32(o.tobytes()) == int(gold["obs_crc"][i]), f"step {i}: observation differs from the reference"
        if i in infos:  # the dict the reference emitted at this step (done / every 10,000 steps), environment.py:1620-1810
            handle.get_info(info_row)
            wram = handle.read_mem(0, 0xD700, 0x200)
            mine = build_info(to_host(info_row)[0], lambda a: int(wram[a - 0xD700]), counts_map=handle.counts_map(0))
            assert info_fingerprint(mine) == infos[i], f"step {i}: info dict differs from the reference's"
        if i % 25 == 0 or i == len(gold["actions"]) - 1:
            sha = np.frombuffer(hashlib.sha256(handle.save_state(0)).digest(), dtype=np.uint8)
            assert np.array_equal(sha, gold["state_sha"][i]), f"step {i}: emulator state differs (RAM side effects / emulation)"
    assert np.array_equal(to_host(obs).reshape(72, 80, 4), gold["last_obs"])


def load_wrapper_sweep():
    """ref_wrapper_sweep.npz with its 264 save-states unpacked.  They are stored as one xz stream (`states_xz`): the
    reference's checkpoints share most of their bytes, which xz finds and the npz's deflate does not (0.25 MB vs 2.5 MB)."""
    gold = dict(np.load(GOLDEN / "ref_wrapper_sweep.npz"))
    gold["states"] = np.frombuffer(lzma.decompress(gold.pop("states_xz").tobytes()), dtype=np.uint8).reshape(len(gold["names"]), -1)
    return gold


def replay_wrapper_sweep(handle, gold, to_dev=lambda a: a, to_host=lambda a: a):
    """ref_wrapper_sweep.npz (all 264 reference save-states x 6 steps of the unmodified reference wrapper) replayed as ONE
    batch: env i starts from state i.  `handle` has 264 envs."""
    n = len(gold["names"])
    for i in range(n):
        handle.set_initial_template(handle.add_state_template(gold["states"][i].tobytes()), np.array([i], dtype=np.int32))
    obs = to_dev(np.zeros((n, _capi.OBS_BYTES), dtype=np.uint8))
    rew = to_dev(np.zeros(n, dtype=np.float64))
    done = to_dev(np.zeros(n, dtype=np.uint8))
    handle.reset(obs, max_episode_steps=int(gold["max_episode_steps"]))
    o = to_host(obs)
    for i in range(n):
        assert zlib.crc32(o[i].tobytes()) == int(gold["reset_obs_crc"][i]), f"{gold['names'][i]}: reset observation differs from the reference"
    for t in range(gold["actions"].shape[1]):
        handle.step(to_dev(np.ascontiguousarray(gold["actions"][:, t])), obs, rew, done)
        r, d, o = to_host(rew), to_host(done), to_host(obs)
        bad = np.nonzero(r != gold["rewards"][:, t])[0]
        assert bad.size == 0, f"step {t}: reward differs from the reference for {[str(gold['names'][i]) for i in bad[:5]]}"
        assert np.array_equal(d, gold["dones"][:, t]), f"step {t}: done differs"
        for i in range(n):
            assert zlib.crc32(o[i].tobytes()) == int(gold["obs_crc"][i, t]), f"step {t}: {gold['names'][i]}: observation differs from the reference"
    for i in range(n):
        sha = np.frombuffer(hashlib.sha256(handle.save_state(i)).digest(), dtype=np.uint8)
        assert np.array_equal(sha, gold["state_sha"][i]), f"{gold['names'][i]}: emulator state differs after the replay"


def ppu_kat_blob(base_blob: bytes, kat, i: int) -> bytes:
    st = parse_state(base_blob)
    st.raw["vram"] = kat["vram"][i]
    st.raw["oam"] = kat["oam"][i]
    st.raw["lcd_regs"] = kat["lcd_regs"][i]
    st.raw["scanline_params"] = kat["scanline_params"][i]
    return serialize_state(st)


def ppu_kat_expected_screen(kat, i: int) -> bytes:
    bits = np.unpackbits(kat["fb2"][i]).reshape(-1, 2)
    shades = bits[:, 0] * 2 + bits[:, 1]
    return SHADE_WORDS[shades].tobytes()


def check_ppu_kat(handle, kat):
    base = handle.save_state(0)
    off, ln = field_offsets(9)["screen"]
    for i in range(len(kat["names"])):
        tid = handle.add_state_template(ppu_kat_blob(base, kat, i))
        handle.load_template(tid)
        handle.debug_render_frame(0)
        got = handle.save_state(0)[off : off + ln]
        assert got == ppu_kat_expected_screen(kat, i), f"PPU KAT {kat['names'][i]}: framebuffer differs from PyBoy's"
