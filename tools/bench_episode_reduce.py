#!/usr/bin/env python
"""Cost of the episode-end reductions a trainer logs: the exploration-map sum (gbenv_counts_map_sum) and the masked
info sum (gbenv_reduce_info_masked), against the per-env path they replace (gbenv_counts_map per env + a host sum).

For each batch size: n envs of the synthetic `pokelike` ROM boot for 60 frames, are reset, and take --steps random-action
steps (seeded), which fills their heat maps; then each call is timed with CUDA events over --reps calls, both back to back
(the directory and the blocks then come from L2 after the first call) and with the L2 overwritten by a 256 MiB memset
before every timed call.  The per-env path is timed with a host clock over a sample of envs (gbenv_counts_map ends in a
stream synchronise) and reported per env.  The card's name and power limit are read in the same run.

usage: tools/bench_episode_reduce.py [--envs 4096 32768] [--steps 200] [--reps 200] [--sample 64] [--out FILE]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402
from pokegym_b200 import _capi  # noqa: E402
from pokegym_b200.tools import synth_rom  # noqa: E402

DIR_BYTES_PER_ENV = 28 * 28 * 4  # heat-map directory entries read per env: 3,136 B


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers below still stand; say where the card data is missing
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def time_events(fn, reps, flush=None):
    """mean device ms of fn() over reps calls; with `flush`, it runs before each call, outside the timed window"""
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(5):  # warm-up
        fn()
    if flush is None:
        torch.cuda.synchronize()
        start.record()
        for _ in range(reps):
            fn()
        end.record()
        end.synchronize()
        return start.elapsed_time(end) / reps
    total = 0.0
    for _ in range(reps):
        flush()
        start.record()
        fn()
        end.record()
        end.synchronize()
        total += start.elapsed_time(end)
    return total / reps


def run(n, steps, reps, sample, lib, rom, scratch):
    dev = torch.device("cuda", 0)
    h = _capi.Handle(lib, n, rom, device_id=0)
    h.tick(60, True)
    obs = torch.zeros((n, _capi.OBS_BYTES), dtype=torch.uint8, device=dev)
    rew = torch.zeros(n, dtype=torch.float64, device=dev)
    done = torch.zeros(n, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    acts = torch.randint(0, 8, (steps, n), generator=gen, device=dev, dtype=torch.uint8)
    h.reset(obs)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for s in range(steps):
        h.step(acts[s], obs, rew, done)
    t1.record()
    h.check()
    step_ms = t0.elapsed_time(t1) / steps

    msum = torch.empty((_capi.COUNTS_H, _capi.COUNTS_W), dtype=torch.int64, device=dev)
    isum = torch.empty(_capi.INFO_SCALARS, dtype=torch.float64, device=dev)
    half = (torch.rand(n, generator=gen, device=dev) < 0.5).to(torch.uint8)
    flush = lambda: scratch.zero_()  # noqa: E731
    res = {"envs": n, "populate": f"tick 60 frames, reset, {steps} steps of seeded random actions (pokelike ROM)",
           "step_ms": round(step_ms, 3), "directory_bytes": n * DIR_BYTES_PER_ENV, "masked_envs_half": int(half.sum())}
    h.counts_map_sum(msum)
    full = msum.cpu().numpy()
    res["map_sum_nonzero_cells"] = int((full != 0).sum())
    res["map_sum_total"] = int(full.sum())
    for name, fn in (("counts_map_sum_all", lambda: h.counts_map_sum(msum)),
                     ("counts_map_sum_half", lambda: h.counts_map_sum(msum, half)),
                     ("reduce_info_masked_half", lambda: h.reduce_info_masked(isum, half)),
                     ("reduce_info_all", lambda: h.reduce_info(isum))):
        res[name + "_ms_l2_warm"] = round(time_events(fn, reps), 4)
        res[name + "_ms_l2_flushed"] = round(time_events(fn, max(reps // 4, 10), flush), 4)

    # the per-env path: one synchronous gather + 774 KB copy per env, summed on the host
    ids = np.linspace(0, n - 1, sample).astype(int)
    total = np.zeros((_capi.COUNTS_H, _capi.COUNTS_W), np.int64)
    h.counts_map(int(ids[0]))
    c0 = time.perf_counter()
    for e in ids:
        total += h.counts_map(int(e))
    per_env_ms = 1000 * (time.perf_counter() - c0) / sample
    res["per_env_counts_map_ms"] = round(per_env_ms, 4)
    res["per_env_path_all_envs_ms_extrapolated"] = round(per_env_ms * n, 1)
    sel = torch.zeros(n, dtype=torch.uint8, device=dev)
    sel[torch.from_numpy(ids).to(dev)] = 1
    h.counts_map_sum(msum, sel)
    res["sample_sum_matches_per_env_path"] = bool(np.array_equal(msum.cpu().numpy(), total))
    h.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 32768])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--sample", type=int, default=64)
    ap.add_argument("--out", type=Path)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_episode_reduce.py measures on a CUDA device; none found")
    lib = _capi.GbEnvLib(g.build_cuda())
    rom = synth_rom.build_pokelike_rom()
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > the 126 MB L2
    out = {"card": card(), "steps": a.steps, "reps": a.reps, "runs": [run(n, a.steps, a.reps, a.sample, lib, rom, scratch) for n in a.envs]}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
