#!/usr/bin/env python
"""Packed observations (obs_format="packed", gbenv_step_packed) against the reference format: step throughput, the cost of
the observation writer alone, the cost of decoding a rollout slot, and rollout memory.

* env-steps/s: EnvGroups of the synthetic `pokelike` ROM booted for 60 frames (bench.py's default start), reference and
  packed built side by side and timed in alternated windows (--runs each), with device-resident random actions and the
  observations written into one slot, as bench.py does.  Batches: 4,096 envs as two groups and as one, 32,768, and one full
  wave of resident envs (SMs x 640: 94,720 on a 148-SM B200).  Each window follows --preroll untimed steps of its own.
* observation writer alone: k_wrap_obs vs k_obs_pack, launched alone on the same synthetic batch by tools/obs_kernels.cu
  (compiled here into a temporary directory) and timed with CUDA events, the L2 overwritten by a 256 MiB memset before every
  timed launch.  Every obs row has a bitmap row to read there (the most work either kernel can have).
* unpack_obs of one ring slot (the packed rows of the batch after the timed steps) with the L2 overwritten the same way.
* rollout bytes at T = 32: computed from the row sizes, not measured.
The card's name and power limit are read in the same run.

usage: tools/bench_obs_packed.py [--runs 2] [--out profiles/obs_packed.json]
"""
import argparse
import ctypes
import json
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402
from bench_episode_reduce import card, time_events  # noqa: E402
from pokegym_b200 import _capi  # noqa: E402
from pokegym_b200.groups import EnvGroups  # noqa: E402
from pokegym_b200.tools import synth_rom  # noqa: E402

T_RING = 32


def obs_kernels_lib(tmp):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out = Path(tmp) / "libobs_kernels.so"
    subprocess.run([nvcc, *g.NVCC_FLAGS, "-o", str(out), str(ROOT / "tools" / "obs_kernels.cu")], check=True)
    lib = ctypes.CDLL(str(out))
    lib.obs_kernel_ms.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
    return lib


def make(lib, rom, n, groups, fmt):
    eg = EnvGroups(lib, n, rom, n_groups=groups, obs_format=fmt)
    eg.for_each(lambda h, gi, st: h.tick(60, True, stream=st))
    row = _capi.OBS_PACKED_BYTES if fmt == "packed" else _capi.OBS_BYTES
    bufs = (torch.zeros((n, row), dtype=torch.uint8, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda"),
            torch.zeros(n, dtype=torch.uint8, device="cuda"))
    eg.reset(bufs[0])
    return eg, bufs


def window(eg, bufs, actions, steps):
    obs, rew, done = bufs
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        eg.step(actions[k % len(actions)], obs, rew, done, join=True)
    torch.cuda.synchronize()
    return eg.num_envs * steps / (time.perf_counter() - t0)


def throughput(lib, rom, n, groups, steps, preroll, runs):
    gen = torch.Generator(device="cuda").manual_seed(n)
    actions = [torch.randint(0, 8, (n,), generator=gen, device="cuda", dtype=torch.uint8) for _ in range(16)]
    made = {fmt: make(lib, rom, n, groups, fmt) for fmt in ("reference", "packed")}
    rates = {fmt: [] for fmt in made}
    for _ in range(runs):
        for fmt, (eg, bufs) in made.items():
            window(eg, bufs, actions, preroll)
            rates[fmt].append(round(window(eg, bufs, actions, steps)))
    packed_rows = made["packed"][1][0]
    res = {"envs": n, "groups": groups, "timed_steps": steps, "preroll_steps": preroll,
           "env_steps_per_s": rates, "packed_over_reference": round(sum(rates["packed"]) / sum(rates["reference"]), 4)}
    for eg, _ in made.values():
        eg.handles[0].check()
    return res, made, packed_rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "obs_packed.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    g.build()
    lib = _capi.GbEnvLib(_capi.DEFAULT_LIB)
    rom = synth_rom.build_pokelike_rom()
    full_wave = torch.cuda.get_device_properties(0).multi_processor_count * 20 * 32
    rec = {"card": card(), "rom": "pokelike (synthetic), booted for 60 frames", "rollout_T": T_RING}
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    flush = lambda: scratch.zero_()  # noqa: E731
    rec["steps"], rec["unpack_one_ring_slot"] = [], []
    for n, groups, steps, preroll in ((4096, 2, 100, 40), (4096, 1, 100, 40), (32768, 1, 30, 10), (full_wave, 1, 12, 4)):
        res, made, packed_rows = throughput(lib, rom, n, groups, steps, preroll, args.runs)
        print(json.dumps(res), flush=True)
        rec["steps"].append(res)
        if groups == 1 and n in (4096, 32768):
            h = made["packed"][0].handles[0]
            out = torch.empty((n, _capi.OBS_BYTES), dtype=torch.uint8, device="cuda")
            ms = time_events(lambda: h.unpack_obs(packed_rows, out), args.reps, flush)
            moved = n * (_capi.OBS_PACKED_BYTES + _capi.OBS_BYTES)
            rec["unpack_one_ring_slot"].append({"envs": n, "ms_l2_flushed": round(ms, 4), "bytes_moved": moved,
                                                "gb_per_s": round(moved / (ms * 1e-3) / 1e9, 1)})
            print(json.dumps(rec["unpack_one_ring_slot"][-1]), flush=True)
        for eg, _ in made.values():
            eg.close()
        del made, packed_rows
        torch.cuda.empty_cache()
    with tempfile.TemporaryDirectory() as tmp:
        klib = obs_kernels_lib(tmp)
        rec["obs_writer_alone"] = []
        for n in (4096, 32768):
            ms = (ctypes.c_float * 2)()
            assert klib.obs_kernel_ms(n, args.reps, ms) == 0
            r = {"envs": n, "k_wrap_obs_ms": round(ms[0], 4), "k_obs_pack_ms": round(ms[1], 4),
                 "k_wrap_obs_bytes_written": n * _capi.OBS_BYTES, "k_obs_pack_bytes_written": n * _capi.OBS_PACKED_BYTES}
            print(json.dumps(r), flush=True)
            rec["obs_writer_alone"].append(r)
    rec["rollout_bytes_T32"] = [{"envs": n, "reference": n * _capi.OBS_BYTES * T_RING, "packed": n * _capi.OBS_PACKED_BYTES * T_RING}
                                for n in (4096, 32768, full_wave)]
    rec["notes"] = ("env-steps/s: EnvGroups step with join, obs into one device slot, reference and packed alternated in one "
                    "process; obs writer alone: synthetic batch, every row with a bitmap row, L2 overwritten before every launch; "
                    "rollout bytes computed, not measured")
    Path(args.out).write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
