#!/usr/bin/env python
"""Cost of the complete episode-end info dicts of a whole batch: gbenv_event_flags (k_event_flags), the masked flag counts
(VecEnvironment.event_counts) and VecEnvironment.episode_infos, against the per-env path they replace.

For each batch size: a VecEnvironment of n envs of the synthetic `pokelike` ROM boots, is reset, and takes --steps
random-action steps (seeded).  Then
  * kernel: gbenv_event_flags over all envs (NULL ids), CUDA events over --reps launches, with the L2 overwritten by a
    256 MiB memset before every timed launch, and back to back (L2 warm) for comparison;
  * counts: event_counts(mask) with half the envs in the mask, CUDA events, L2 overwritten the same way;
  * end to end: host wall time of episode_infos(all envs), which ends in a device-to-host copy (a synchronise);
  * old path: the per-env full_info as it was before gbenv_event_flags (info rows to the host, gbenv_read_mem of
    0xD700-0xD8FF, gbenv_counts_map, build_info) and full_info as it is now, host wall time over --sample envs, per env.
    Any figure for all envs is in a field named `..._extrapolated`.
The card's name and power limit are read in the same run.

usage: tools/bench_episode_infos.py [--envs 4096 32768] [--steps 200] [--reps 200] [--sample 32] [--out FILE]
"""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402
from pokegym_b200 import VecEnvironment, _capi  # noqa: E402
from pokegym_b200 import info as I  # noqa: E402
from pokegym_b200.tools import synth_rom  # noqa: E402

sys.path.insert(0, str(ROOT / "tools"))
from bench_episode_reduce import card, time_events  # noqa: E402


def old_full_info(vec, e):
    """full_info before gbenv_event_flags: three synchronous round trips per env"""
    row = vec.info()[e].cpu().numpy()
    wram = vec.handle.read_mem(e, 0xD700, 0x200)
    cm = vec.handle.counts_map(e).astype(np.float64)
    return I.build_info(row, lambda a: int(wram[a - 0xD700]), counts_map=cm, reward_scale=vec.reward_scale)


def run(n, steps, reps, sample, rom, scratch):
    dev = torch.device("cuda", 0)
    vec = VecEnvironment(n, rom, device=dev)
    vec.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    acts = torch.randint(0, 8, (steps, n), generator=gen, device=dev, dtype=torch.uint8)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for s in range(steps):
        vec.step(acts[s])
    t1.record()
    vec.handle.check()
    res = {"envs": n, "populate": f"boot 60 frames, reset, {steps} steps of seeded random actions (pokelike ROM)",
           "step_ms": round(t0.elapsed_time(t1) / steps, 3)}

    flags = torch.empty((n, _capi.EVENT_WORDS), dtype=torch.int32, device=dev)
    counts = torch.empty(_capi.EVENT_FLAGS, dtype=torch.int64, device=dev)
    half = (torch.rand(n, generator=gen, device=dev) < 0.5).to(torch.uint8)
    flush = lambda: scratch.zero_()  # noqa: E731
    kernel = lambda: vec.handle.event_flags(flags, stream=vec._stream())  # noqa: E731
    res["event_flags_kernel_ms_l2_flushed"] = round(time_events(kernel, reps, flush), 4)
    res["event_flags_kernel_ms_l2_warm"] = round(time_events(kernel, reps), 4)
    res["event_flags_bytes_written"] = n * _capi.EVENT_WORDS * 4
    res["event_flags_lines_read"] = (n // 32) * 17  # 17 distinct WRAM words, one 128-byte line per word per 32-env tile
    res["event_counts_half_ms_l2_flushed"] = round(time_events(lambda: vec.event_counts(half, out=counts), max(reps // 4, 10), flush), 4)
    res["envs_with_a_flag_set"] = int((flags != 0).any(1).sum())
    res["flags_set_total"] = int(vec.event_counts(out=counts).sum())

    everything = torch.ones(n, dtype=torch.uint8, device=dev)
    vec.episode_infos(everything)  # warm-up
    walls = []
    for _ in range(3):
        torch.cuda.synchronize()
        c0 = time.perf_counter()
        infos = vec.episode_infos(everything)
        torch.cuda.synchronize()
        walls.append(1000 * (time.perf_counter() - c0))
    res["episode_infos_all_envs_ms"] = [round(w, 1) for w in walls]
    res["episode_infos_dicts"] = len(infos)

    ids = np.linspace(0, n - 1, sample).astype(int)
    for name, fn in (("old_full_info", lambda e: old_full_info(vec, e)), ("full_info", vec.full_info)):
        fn(int(ids[0]))
        c0 = time.perf_counter()
        for e in ids:
            fn(int(e))
        per_env = 1000 * (time.perf_counter() - c0) / sample
        res[f"{name}_per_env_ms"] = round(per_env, 3)
        res[f"{name}_all_envs_ms_extrapolated"] = round(per_env * n, 1)
    res["per_env_sample"] = sample

    def strip(d):
        d = dict(d, pokemon_exploration_map=None)
        d["stats"] = dict(d["stats"], pokemon_exploration_map=None)
        return d

    res["sample_matches_old_path"] = all(infos[int(e)] == strip(old_full_info(vec, int(e))) for e in ids)
    vec.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 32768])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--sample", type=int, default=32)
    ap.add_argument("--out", type=Path)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_episode_infos.py measures on a CUDA device; none found")
    g.build_cuda()
    rom = synth_rom.build_pokelike_rom()
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > the 126 MB L2
    out = {"card": card(), "steps": a.steps, "reps": a.reps, "runs": [run(n, a.steps, a.reps, a.sample, rom, scratch) for n in a.envs]}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
