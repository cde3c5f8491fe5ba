#!/usr/bin/env python
"""Cost of batched frame capture (gbenv_capture_frames) and decode (gbenv_frames_to_rgb), against the per-env path they
replace (gbenv_screen per env), and the effect of a FrameRecorder on VecEnvironment step throughput.

For each batch size: n envs of the synthetic `pokelike` ROM boot for 60 frames, are reset and take --steps random-action
steps (seeded).  Captures of 16, 256 (spread evenly over the batch, so each entry is in a different 32-env tile: reads are
not coalesced across entries) and all envs (NULL ids: coalesced reads) are timed with CUDA events over --reps launches, back
to back (L2 warm) and with the L2 overwritten by a 256 MiB memset before each timed launch.  GB/s counts the bytes the kernel
must move: each frame's 5,760 B read once and written once.  The decode of 1,000 frames is timed the same way, grey and RGB
(bytes: 5,760 read + 23,040 x channels written per frame).  gbenv_screen is timed with a host clock around its synchronous
calls on the same 16 envs.  Step throughput: VecEnvironment at --step-envs envs, without a recorder and with a 16-env
recorder, in --pairs alternated runs of --step-steps steps each.  The card's name and power limit are read in the same run.

usage: tools/bench_frames.py [--envs 4096 32768] [--steps 30] [--reps 200] [--step-envs 4096] [--out FILE]
"""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402
from bench_episode_reduce import card, time_events  # noqa: E402
from pokegym_b200 import _capi  # noqa: E402
from pokegym_b200.tools import synth_rom  # noqa: E402

FRAME_BYTES = _capi.FRAME_WORDS * 4
PIXELS = _capi.SCREEN_H * _capi.SCREEN_W


def gbps(nbytes, ms):
    return round(nbytes / (ms * 1e-3) / 1e9, 1)


def run(n, steps, reps, lib, rom, scratch):
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
    flush = lambda: scratch.zero_()  # noqa: E731
    res = {"envs": n, "populate": f"tick 60 frames, reset, {steps} steps of seeded random actions (pokelike ROM)"}
    frames = torch.empty((n, _capi.FRAME_WORDS), dtype=torch.int32, device=dev)
    for k in (16, 256, n):
        ids = None if k == n else torch.from_numpy(np.linspace(0, n - 1, k).astype(np.int32)).to(dev)
        fn = lambda: h.capture_frames(frames[:k], ids)  # noqa: E731
        moved = 2 * k * FRAME_BYTES
        warm, cold = time_events(fn, reps), time_events(fn, max(reps // 4, 10), flush)
        name = f"capture_{'all' if k == n else k}"
        res[name] = {"ids": "NULL (all envs)" if ids is None else "spread evenly", "bytes_moved": moved, "ms_l2_warm": round(warm, 4),
                     "gbps_l2_warm": gbps(moved, warm), "ms_l2_flushed": round(cold, 4), "gbps_l2_flushed": gbps(moved, cold)}
    sample = np.linspace(0, n - 1, 16).astype(int)
    h.screen(int(sample[0]))
    c0 = time.perf_counter()
    for e in sample:
        h.screen(int(e))
    res["per_env_screen_x16_ms"] = round(1000 * (time.perf_counter() - c0), 3)
    torch.cuda.synchronize()
    c0 = time.perf_counter()
    h.capture_frames(frames[:16], torch.from_numpy(sample.astype(np.int32)).to(dev))
    torch.cuda.synchronize()
    res["capture_16_host_ms_incl_sync"] = round(1000 * (time.perf_counter() - c0), 3)
    h.close()
    return res


def decode(lib, rom, reps, scratch, n_frames=1000):
    dev = torch.device("cuda", 0)
    h = _capi.Handle(lib, 1, rom, device_id=0)
    frames = torch.randint(-2**31, 2**31 - 1, (n_frames, _capi.FRAME_WORDS), dtype=torch.int32, device=dev)
    res = {"frames": n_frames}
    for ch, name in ((1, "grey"), (3, "rgb")):
        out = torch.empty((n_frames, _capi.SCREEN_H, _capi.SCREEN_W, ch), dtype=torch.uint8, device=dev)
        fn = lambda: h.frames_to_rgb(frames, out, ch)  # noqa: E731
        moved = n_frames * (FRAME_BYTES + PIXELS * ch)
        warm, cold = time_events(fn, reps), time_events(fn, max(reps // 4, 10), lambda: scratch.zero_())
        res[name] = {"bytes_moved": moved, "ms_l2_warm": round(warm, 4), "gbps_l2_warm": gbps(moved, warm), "ms_l2_flushed": round(cold, 4),
                     "gbps_l2_flushed": gbps(moved, cold)}
    h.close()
    return res


def step_throughput(n, steps, pairs, rom):
    """env-steps/s of VecEnvironment.step, without and with a 16-env recorder, alternated."""
    from pokegym_b200 import VecEnvironment

    dev = torch.device("cuda", 0)
    vec = VecEnvironment(n, rom, auto_reset=True)
    vec.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(2)
    acts = torch.randint(0, 8, (steps, n), generator=gen, device=dev, dtype=torch.uint8)
    ids = np.linspace(0, n - 1, 16).astype(np.int32)

    def one(recorder):
        vec.record_frames(ids, capacity=steps) if recorder else vec.record_frames(None)
        for s in range(10):  # warm-up
            vec.step(acts[s])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(steps):
            vec.step(acts[s])
        torch.cuda.synchronize()
        return round(n * steps / (time.perf_counter() - t0), 1)

    runs = {"none": [], "recorder_16": []}
    for _ in range(pairs):
        runs["none"].append(one(False))
        runs["recorder_16"].append(one(True))
    vec.close()
    return {"envs": n, "steps_per_run": steps, "env_steps_per_s": runs}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 32768])
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--step-envs", type=int, default=4096)
    ap.add_argument("--step-steps", type=int, default=150)
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--out", type=Path)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_frames.py measures on a CUDA device; none found")
    lib = _capi.GbEnvLib(g.build_cuda())
    rom = synth_rom.build_pokelike_rom()
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > the 126 MB L2
    out = {"card": card(), "reps": a.reps, "capture": [run(n, a.steps, a.reps, lib, rom, scratch) for n in a.envs],
           "decode": decode(lib, rom, a.reps, scratch), "step": step_throughput(a.step_envs, a.step_steps, a.pairs, rom)}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
