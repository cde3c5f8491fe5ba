#!/usr/bin/env python
"""Cost of batched save-states (gbenv_save_states) against the per-env call (gbenv_save_state) it complements.

For each batch size: n envs of the synthetic `pokelike` ROM boot for 60 frames, are reset and take --steps random-action
steps (seeded).  gbenv_save_states of all envs (NULL ids) is timed with CUDA events over --reps launches back to back; the
output alone (n x 142,610 B: 584 MB at 4,096 envs, 4.7 GB at 32,768) is larger than the 126 MB L2, so the launches do not
run from a warm cache.  Bytes: n x 142,610 written, and n x 56,640 read (every word of the env's state once; the words a
16-byte unit at a chunk edge shares with the next chunk are read twice, a few hundred bytes per env, not counted).  GB/s is
those bytes over the kernel time; the fraction is of the HBM3e data-sheet rate for one B200, 7.7 TB/s.  The kernel does no
arithmetic to speak of, so memory bandwidth is its bound.  gbenv_save_state is timed for comparison with a host clock
around --single consecutive calls (each one launch, a 142,610 B copy to pageable host memory and a synchronise), per env.
The card's name and power limit are read in the same run.

usage: tools/bench_save_states.py [--envs 4096 32768] [--steps 30] [--reps 50] [--single 256] [--out profiles/save_states.json]
"""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402
from bench_episode_reduce import card, time_events  # noqa: E402
from pokegym_b200 import _capi  # noqa: E402
from pokegym_b200.tools import synth_rom  # noqa: E402

STATE_READ_BYTES = (0x4200 + 0x8000 + 1440 * 4 + 288 * 4 + 16 * 4)  # IMG_WORDS * 4: mem, cart RAM, framebuffer, scanlines, registers
HBM_TBPS = 7.7


def run(n, steps, reps, single, lib, rom):
    dev = torch.device("cuda", 0)
    h = _capi.Handle(lib, n, rom, device_id=0)
    h.tick(60, True)
    obs = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device=dev)
    rew = torch.zeros(n, dtype=torch.float64, device=dev)
    done = torch.zeros(n, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    h.reset(obs)
    for _ in range(steps):
        h.step(torch.randint(0, 8, (n,), generator=gen, device=dev, dtype=torch.uint8), obs, rew, done)
    h.check()
    del obs
    blobs = torch.empty((n, _capi.STATE_BYTES), dtype=torch.uint8, device=dev)
    ms = time_events(lambda: h.save_states(blobs), reps)
    written, read = n * _capi.STATE_BYTES, n * STATE_READ_BYTES
    rate = (written + read) / (ms * 1e-3) / 1e9
    res = {"envs": n, "populate": f"tick 60 frames, reset, {steps} steps of seeded random actions (pokelike ROM)",
           "save_states_all": {"ids": "NULL (all envs)", "reps": reps, "ms": round(ms, 4), "bytes_written": written, "bytes_read": read,
                               "gbps": round(rate, 1), "fraction_of_hbm_7.7TBps": round(rate / (HBM_TBPS * 1e3), 3), "bound": "HBM bandwidth",
                               "us_per_env": round(1000 * ms / n, 4)}}
    k = min(single, n)
    h.save_state(0)
    c0 = time.perf_counter()
    for e in range(k):
        h.save_state(e)
    h.sync()
    res["save_state_loop"] = {"envs": k, "ms_total": round(1000 * (time.perf_counter() - c0), 3),
                              "us_per_env": round(1e6 * (time.perf_counter() - c0) / k, 2)}
    torch.cuda.synchronize()
    row0 = blobs[0].cpu().numpy().tobytes()
    assert row0 == h.save_state(0), "batched row differs from gbenv_save_state"
    h.close()
    del blobs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 32768])
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--single", type=int, default=256)
    ap.add_argument("--out", type=Path, default=ROOT / "profiles" / "save_states.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_save_states.py measures on a CUDA device; none found")
    lib = _capi.GbEnvLib(g.build_cuda())
    rom = synth_rom.build_pokelike_rom()
    out = {"card": card(), "runs": [run(n, a.steps, a.reps, a.single, lib, rom) for n in a.envs]}
    text = json.dumps(out, indent=1)
    print(text)
    a.out.parent.mkdir(parents=True, exist_ok=True)
    a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
