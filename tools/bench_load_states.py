#!/usr/bin/env python
"""Cost of batched load-states (gbenv_load_states) against the per-row path it replaces.

For each batch size: n envs of the synthetic `pokelike` ROM boot for 60 frames, are reset and take --steps random-action
steps (seeded); save_states writes all their rows, and gbenv_load_states of all envs from those rows (NULL ids, status
reported) is timed with CUDA events over --reps launches back to back.  The rows alone (n x 142,610 B: 584 MB at 4,096 envs,
4.7 GB at 32,768) are larger than the 126 MB L2, so the launches do not run from a warm cache.  Bytes counted per env:
142,610 read by the load pass (every row byte once; the few hundred bytes of 16-byte units that two chunks share are not
counted), 92,160 re-read by the check pass (the screen section), and 56,640 written (the env's image: every word once).
GB/s is those bytes over the time of both kernels; the fraction is of the HBM3e data-sheet rate for one B200, 7.7 TB/s.
The kernels do no arithmetic to speak of, so memory bandwidth is their bound.  The path it replaces is timed for up to
--single rows with a host clock: copy the row to the host, gbenv_add_state_template (host parse, allocation, synchronous
upload), gbenv_load_template (synchronous).  The card's name and power limit are read in the same run.

usage: tools/bench_load_states.py [--envs 4096 32768] [--steps 30] [--reps 30] [--single 1024] [--out profiles/load_states.json]
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
from bench_save_states import STATE_READ_BYTES  # noqa: E402
from pokegym_b200 import _capi  # noqa: E402
from pokegym_b200.tools import synth_rom  # noqa: E402

SCREEN_BYTES = 144 * 160 * 4
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
    h.save_states(blobs)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    ms = time_events(lambda: h.load_states(blobs, status=status), reps)
    torch.cuda.synchronize()
    assert bool((status == 0).all()), "a saved row was rejected"
    again = torch.empty_like(blobs)
    h.save_states(again)
    assert torch.equal(again, blobs), "loading the envs' own rows changed them"
    del again
    read, reread, written = n * _capi.STATE_BYTES, n * SCREEN_BYTES, n * STATE_READ_BYTES
    rate = (read + reread + written) / (ms * 1e-3) / 1e9
    res = {"envs": n, "populate": f"tick 60 frames, reset, {steps} steps of seeded random actions (pokelike ROM); rows from save_states",
           "load_states_all": {"ids": "NULL (all envs)", "reps": reps, "ms": round(ms, 4), "bytes_read_rows": read,
                               "bytes_reread_screen_check": reread, "bytes_written": written, "gbps": round(rate, 1),
                               "fraction_of_hbm_7.7TBps": round(rate / (HBM_TBPS * 1e3), 3), "bound": "HBM bandwidth",
                               "us_per_env": round(1000 * ms / n, 4)}}
    k = min(single, n)
    torch.cuda.synchronize()
    c0 = time.perf_counter()
    for e in range(k):  # what a caller had to do per row before gbenv_load_states (each call takes one template slot)
        row = blobs[e].cpu().numpy().tobytes()
        h.load_template(h.add_state_template(row), [e])
    h.sync()
    dt = time.perf_counter() - c0
    res["per_row_path"] = {"rows": k, "steps": "row to host, add_state_template, load_template", "ms_total": round(1000 * dt, 3),
                           "us_per_row": round(1e6 * dt / k, 2)}
    h.close()
    del blobs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 32768])
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--single", type=int, default=1024)
    ap.add_argument("--out", type=Path, default=ROOT / "profiles" / "load_states.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_load_states.py measures on a CUDA device; none found")
    lib = _capi.GbEnvLib(g.build_cuda())
    rom = synth_rom.build_pokelike_rom()
    out = {"card": card(), "runs": [run(n, a.steps, a.reps, a.single, lib, rom) for n in a.envs]}
    text = json.dumps(out, indent=1)
    print(text)
    a.out.parent.mkdir(parents=True, exist_ok=True)
    a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
