#!/usr/bin/env python
"""Class mix of the benchmark workloads (CPU only; input of tools/gen_classes.sh).

Runs the device headers on the host with -DGB_SLOT_TRACE (tests/hostsim, the tracing build of tools/trace_convergence.py)
over the workloads bench.py times -- the pokelike, busy and pokelike_timer ROMs booted for 60 frames, and the pokelike
ROM from the 40 mixed reference save-states -- and counts how often the fast loop executes each (handler, operand flags)
pair.  Every workload weighs the same (its counts are normalised to 1,000,000 instructions).  Writes one line per pair,
"handler flags count", hottest first, to tools/class_counts.txt: tools/gen_classes.cpp orders the class ids and shapes the
single-lane dispatch from it.

usage: python tools/class_mix.py [--envs 8] [--steps 6]
"""
import argparse
import ctypes as C
import sys
from collections import Counter
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT.parent))
sys.path.insert(0, str(ROOT.parent / "tests" / "hostsim"))
sys.path.insert(0, str(ROOT))

WORKLOADS = (("pokelike", False), ("busy", False), ("pokelike_timer", False), ("pokelike", True))


def workload_mix(driver, rom, n, steps, mixed):
    hs = driver.HostSim(n, rom)
    hs.dll.hs_slots.restype = C.c_size_t
    hs.dll.hs_slots.argtypes = [C.c_void_p, C.c_size_t]
    if mixed:
        blobs = np.load(ROOT.parent / "tests" / "golden" / "red_states_mixed.npz")["states"]
        for e in range(n):
            hs.load_blob(e, blobs[(5 * e) % len(blobs)].tobytes())
    else:
        hs.tick(60, True)
    hs.dll.hs_slots(None, 0)
    mix = Counter()
    rng = np.random.default_rng(5)
    for _ in range(steps):
        hs.run_action(rng.integers(0, 8, n).astype(np.uint8))
        rec = np.empty(hs.dll.hs_slots(None, 0), dtype=np.uint64)
        hs.dll.hs_slots(rec.ctypes.data, len(rec))
        rec = rec[(rec >> np.uint64(48)) == 0]  # instructions of the fast loop
        key = ((rec >> np.uint64(24)) & np.uint64(0xFF)) << np.uint64(16) | ((rec >> np.uint64(32)) & np.uint64(0xFFF0))
        k, c = np.unique(key, return_counts=True)
        mix.update(dict(zip(k.tolist(), c.tolist())))
    hs.close()
    return mix


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8)
    ap.add_argument("--steps", type=int, default=6)
    args = ap.parse_args()
    import driver
    from trace_convergence import build
    from pokegym_b200.tools import synth_rom

    driver.build = build  # the tracing build
    total = Counter()
    for name, mixed in WORKLOADS:
        fn, kw = synth_rom.rom_catalog()[name]
        mix = workload_mix(driver, fn(**kw), args.envs, args.steps, mixed)
        n = sum(mix.values())
        for k, c in mix.items():
            total[k] += c * 1_000_000 / n
        print(f"{name}{' (mixed states)' if mixed else ''}: {n} instructions", file=sys.stderr)
    with open(ROOT / "class_counts.txt", "w") as f:
        f.write("# handler flags count -- tools/class_mix.py: fast-loop instructions per (handler, operand flags) pair, the benchmark\n"
                f"# workloads weighted equally ({', '.join(n + (' mixed' if m else '') for n, m in WORKLOADS)}; {args.envs} envs x {args.steps} steps each)\n")
        for k, c in sorted(total.items(), key=lambda kv: -kv[1]):
            f.write(f"{k >> 16} 0x{k & 0xFFFF:04x} {round(c)}\n")


if __name__ == "__main__":
    main()
