#!/usr/bin/env python
"""Headline benchmark: env-steps/s of the batched Game Boy environment (24 emulated frames + reward +
observation per env-step), BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu E] [--impl reference] [--config single] [--only-leg NAME]

* one process per GPU; for N > 1 the driver launches this file under torchrun (RANK / LOCAL_RANK /
  WORLD_SIZE / MASTER_* from the environment) and every rank owns E envs (weak scaling, SURVEY.md 8e);
  the only collective is the NCCL all-reduce of the 72-double episode-info vector, once per 32-step rollout
  and at least once inside every timed region.
* `value`   : whole-job env-steps/s with actions already resident in HBM and observations written into a
              device rollout tensor u8[32, E, 72*80*4]; CUDA-event timed, max over ranks.  Before the W
              warm-up steps every env is pre-rolled for PREROLL steps, so that the timed region starts from the
              diverged steady state (envs that start together drift apart for ~150 steps).
* `e2e`     : the same metric through the host-buffer C-ABI calls gbenv_submit_host / gbenv_fetch_host (pinned host
              memory; actions H2D and obs/reward/done D2H inside the timed region, the D2H of step t overlapped
              with the emulation of step t+1 exactly as a vectoriser that double-buffers would).
* `roofline`: algorithmic bytes (57,682 B per env-step, BASELINE.md section 4) of the dominant kernel
              k_run_frames over its CUDA-event duration, against the measured HBM peak.  `issue` is the figure
              that actually bounds this kernel (an interpreter: instruction issue, not bandwidth).
* `legs`    : (1 GPU only) the other workloads SURVEY.md 8d names: 32,768 envs, the 100 %-busy ROM, the TIMA ROM,
              the divergence stress of BASELINE.json config 5 (envs reset from 40 different reference save-states),
              72 envs (README config) and 1 env (config 1, short form; `--config single` runs test.py's full protocol).
* `cpu_baseline` / `--impl reference`: the CPU oracle (a port of the reference's algorithm; PyBoy itself
              cannot be installed here) on the box's host cores, on a bounded sample of the same workload.
* `--dump-outputs DIR`: what the timed path handed its caller at its last step, as float32 / float64 .npy files
              (see dump_outputs), so that two builds can be compared output for output on identical inputs.

The benchmark writes nothing into the repository tree: a library whose sources are newer than the build that
build() left there is rebuilt in a temporary directory.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
SCRATCH = tempfile.TemporaryDirectory(prefix="pokegym-bench-")  # rebuilds of stale libraries; removed at exit

ALGO_BYTES_PER_ENV_STEP = 57_682  # BASELINE.md section 4 / SURVEY.md 8d
ROLLOUT_T = 32
PREROLL = 200  # untimed steps before the warm-up: envs that start from one state need ~150 steps to reach their steady spread
WORKLOAD = "pokelike synthetic ROM (MBC3, ~25% busy frames), random actions, full reward shaping, obs into device rollout u8[32,E,72,80,4]"
MIXED_STATES = ROOT / "tests" / "golden" / "red_states_mixed.npz"


def workload_name(args) -> str:
    from pokegym_b200.tools import synth_rom

    if args.rom == "pokelike" and not args.state:
        return WORKLOAD
    what = f"synthetic ROM '{args.rom}'" if args.rom in synth_rom.rom_catalog() else f"user ROM {Path(args.rom).name}"
    start = f"reset from {Path(args.state).name}" if args.state else "booted for 60 frames"
    return f"{what}, {start}, random actions, full reward shaping, obs into device rollout u8[32,E,72,80,4]"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 10,000 with --config single)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--envs-per-gpu", type=int, default=4096)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rom", default=os.environ.get("POKEGYM_ROM", "pokelike"), help="synthetic ROM name or path to a .gb file")
    ap.add_argument("--state", default=None, help="PyBoy .state file every env resets from (default: boot the ROM for 60 frames)")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--cpu-baseline-seconds", type=float, default=12.0)
    ap.add_argument("--preroll", type=int, default=PREROLL)
    ap.add_argument("--groups", type=int, default=0,
                    help="env groups stepping on separate CUDA streams (pokegym_b200.EnvGroups); 0 = 2 while every env has a warp of its own, else 1")
    ap.add_argument("--legs", default="all", help="'all', 'none' or a comma list of leg names (1 GPU only)")
    ap.add_argument("--only-leg", default=None, help="run one leg alone and print its record (profiling)")
    ap.add_argument("--config", default=None, choices=[None, "single"], help="single: BASELINE.json config 1, the protocol of the reference's test.py")
    ap.add_argument("--also-envs", type=int, default=-1,
                    help="extra single-GPU leg at this env count, reported under 'large_batch' (0 = skip; -1 = one full wave of resident envs)")
    ap.add_argument("--also-steps", type=int, default=12)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the observations, rewards, dones and info sum of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.steps is None and not (args.config == "single" and args.impl == "ours"):  # run_single_config: None = test.py's protocol
        args.steps = 200
    if args.dump_outputs and (args.impl != "ours" or args.config or args.only_leg):
        ap.error("--dump-outputs writes the outputs of the headline run: it does not combine with --impl reference, --config or --only-leg")
    return args


def library(build):
    """Path of the shared library `build` (__graft_entry__.build_cuda or build_oracle) makes: the one build() left in the
    tree while it is current, else a fresh build in SCRATCH."""
    return build(out_dir=SCRATCH.name)


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_hash() -> str:
    """Hash of the CUDA sources: profile-derived constants (profiles/kernel_counters.json) are only reported while they
    describe the kernel that is actually being benchmarked."""
    h = hashlib.sha256()
    for p in sorted((ROOT / "pokegym_b200" / "csrc").glob("*")):
        if p.suffix in (".cu", ".cuh", ".h", ".inc"):
            h.update(p.name.encode())
            h.update(p.read_bytes())
    return h.hexdigest()[:16]


def recorded_counters(name="kernel_counters.json"):
    """ncu-derived per-launch counters of the emulation kernel (tools/summarise_profile.py), or None when they are stale
    (taken from another version of the CUDA sources)."""
    p = ROOT / "profiles" / name
    try:
        d = json.load(open(p))
    except Exception:
        return None
    return d if d.get("kernel_source_hash") == kernel_source_hash() else None


def issue_record(counters, kernel_ms, sm_mhz, n_sms):
    """Instruction-issue view of a launch: SASS warp-instructions per emulated SM83 instruction and lanes active come from a
    committed ncu capture of THIS kernel source (hash-stamped); the rates use this run's kernel time and clock."""
    wi, emu = counters["warp_instructions_per_launch"], counters["emulated_instructions_per_launch"]
    peak = n_sms * 4 * sm_mhz * 1e6
    return {"kernel": counters.get("kernel"), "warp_instr_per_emulated_instr": wi / emu, "thread_instr_per_emulated_instr": wi * counters["lanes_active"] / emu,
            "lanes_active_per_warp_instr": counters["lanes_active"], "warp_instr_per_s": wi / (kernel_ms / 1000.0), "peak_warp_instr_per_s": peak,
            "frac": wi / (kernel_ms / 1000.0) / peak, "ncu_issue_active_pct": counters.get("issue_active_pct"), "ncu_alu_pipe_pct": counters.get("alu_pipe_pct"),
            "ncu_sm_active_share_of_elapsed": counters.get("sm_active_share_of_elapsed"), "source": counters.get("source")}


def tier_b_record():
    """BASELINE.md tier B (the reference's unmodified wrapper over the oracle core, one process per core): measured where the
    reference tree is mounted (tools/cpu_tier_b.py) and quoted from the committed file."""
    for p in sorted((ROOT / "profiles").glob("*_cpu_tier_b.json"), reverse=True):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return None


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampler running during the timed region."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


def build_rom(name: str) -> bytes:
    """`name` is a synthetic ROM of pokegym_b200.tools.synth_rom.rom_catalog() or a path to a user-supplied .gb file
    (BASELINE.json config 1: pokemon_red.gb; no ROM ships with the reference, so the default is synthetic)."""
    from pokegym_b200.tools import synth_rom

    if name in synth_rom.rom_catalog():
        fn, kw = synth_rom.rom_catalog()[name]
        return fn(**kw)
    return Path(name).read_bytes()


def mixed_states():
    """The 40 reference save-states of BASELINE.json config 5 (tools/select_mixed_states.py)."""
    import numpy as np

    return [s.tobytes() for s in np.load(MIXED_STATES)["states"]]


def start_envs(h, state_path, n_envs=None, mixed=False):
    """Every env starts from the same point -- the given PyBoy .state file, or the ROM booted for 60 frames -- or, for the
    divergence stress, env i from reference save-state i mod 40."""
    import numpy as np

    if mixed:
        for k, blob in enumerate(mixed_states()):
            ids = np.arange(k, n_envs, 40, dtype=np.int32)
            if ids.size:
                h.set_initial_template(h.add_state_template(blob), ids)
    elif state_path:
        h.set_initial_template(h.add_state_template(Path(state_path).read_bytes()))
    else:
        h.tick(60, True)


# ------------------------------------------------------------------------------------------------ CPU arm

def oracle_run(rom: bytes, seconds: float, n_envs=None, state_path=None, mixed=False, min_steps=3):
    """CPU oracle (port of the reference path) on all host cores for about `seconds`; returns (value, cores, sample)."""
    import numpy as np

    from pokegym_b200 import _capi
    import __graft_entry__ as g

    lib = _capi.GbEnvLib(library(g.build_oracle), "oracle_")
    cores = os.cpu_count() or 1
    n = n_envs or max(cores * 16, 64)  # >= 16 envs per worker thread: thread start-up is amortised over ~20 ms of work
    h = _capi.Handle(lib, n, rom)
    start_envs(h, state_path, n, mixed)
    obs = np.zeros((n, _capi.OBS_BYTES), dtype=np.uint8)
    rew = np.zeros(n)
    done = np.zeros(n, dtype=np.uint8)
    h.reset(obs)
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 8, (4096, n)).astype(np.uint8)
    for i in range(2):
        h.step(acts[i], obs, rew, done)
    steps, t0 = 0, time.perf_counter()
    while True:
        h.step(acts[(steps + 2) % 4096], obs, rew, done)
        steps += 1
        dt = time.perf_counter() - t0
        if (dt >= seconds and steps >= min_steps) or steps >= 100000:
            break
    h.close()
    return n * steps / dt, cores, f"{n} envs x {steps} env-steps of the same ROM / reset state / action distribution in {dt:.1f} s on {cores} host threads"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  PyBoy (the emulator the reference drives) is an
    un-vendored dependency that cannot be installed here, so this arm times the oracle port on every host core.
    A 'step' is one pass of a bounded sample (16 envs per host thread, repeated so that K steps last >= ~2.5 s whatever K)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np

    from pokegym_b200 import _capi
    import __graft_entry__ as g

    rom = build_rom(args.rom)
    cores = os.cpu_count() or 1
    n = max(cores * 16, 64)
    lib = _capi.GbEnvLib(library(g.build_oracle), "oracle_")
    h = _capi.Handle(lib, n, rom)
    start_envs(h, args.state, n)
    obs = np.zeros((n, _capi.OBS_BYTES), dtype=np.uint8)
    rew = np.zeros(n)
    done = np.zeros(n, dtype=np.uint8)
    h.reset(obs)
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 8, (4096, n)).astype(np.uint8)
    k = 0

    def one_pass():
        nonlocal k
        h.step(acts[k % 4096], obs, rew, done)
        k += 1

    t0 = time.perf_counter()
    for _ in range(3):
        one_pass()
    per_pass = (time.perf_counter() - t0) / 3
    W, K = max(args.warmup, 3), args.steps
    repeats = max(1, int(2.5 / max(per_pass * K, 1e-9) + 0.999))  # env-steps per env inside one timed 'step'
    for _ in range(W):
        one_pass()
    t0 = time.perf_counter()
    for _ in range(K * repeats):
        one_pass()
    dt = time.perf_counter() - t0
    value = n * K * repeats / dt
    sample = f"{n} envs x {repeats} env-steps per step x {K} steps in {dt:.1f} s on {cores} host threads (oracle port; PyBoy + ROM unavailable)"
    line = {
        "impl": "reference", "metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": 1000.0 * dt / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_name(args), "envs_per_step": n * repeats, "act_freq": 24, "rom": args.rom,
                   "note": "bounded sample: each step advances `envs_per_step` env-steps on the host cores"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "frames_per_s": 24 * value,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU legs

def e2e_host_loop(hs, E, n_e2e, world=1, dev=None):
    """The same metric through gbenv_submit_host / gbenv_fetch_host with pinned host buffers: actions H2D and obs / reward / done
    D2H inside the timed region, step t+1 submitted before the results of step t are fetched (two steps in flight), so the
    observation copy overlaps the next emulation kernel -- what a vectoriser that keeps two rollout slots in flight does.
    `hs`: the handles of the env groups (one, or several that share the E envs evenly).
    Returns env-steps/s of this rank's E envs (wall clock around the loop, max over ranks when world > 1)."""
    import torch
    import torch.distributed as dist

    from pokegym_b200 import _capi
    from pokegym_b200.dist import max_over_ranks

    hs = list(hs) if isinstance(hs, (list, tuple)) else [hs]
    G, n = len(hs), E // len(hs)
    act_h = torch.randint(0, 8, (n_e2e + 4, E), dtype=torch.uint8).pin_memory()
    obs_h = [torch.zeros((E, _capi.OBS_BYTES), dtype=torch.uint8).pin_memory() for _ in range(2)]
    rew_h = [torch.zeros(E, dtype=torch.float64).pin_memory() for _ in range(2)]
    done_h = [torch.zeros(E, dtype=torch.uint8).pin_memory() for _ in range(2)]

    def submit(i):
        for g, h in enumerate(hs):
            a, b = g * n, (g + 1) * n
            h.submit_host(act_h[i][a:b].numpy(), obs_h[i % 2][a:b].numpy(), rew_h[i % 2][a:b].numpy(), done_h[i % 2][a:b].numpy())

    def fetch():
        for h in hs:
            h.fetch_host()

    for i in range(3):
        submit(i)
        fetch()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    submit(3)
    for i in range(4, 3 + n_e2e):
        submit(i)  # step i queued behind step i-1 ...
        fetch()    # ... while the results of step i-1 arrive (blocks until they are in the host buffers)
        float(rew_h[(i - 1) % 2][0])  # the caller reads them
    fetch()
    float(rew_h[(2 + n_e2e) % 2][0])
    e2e_s = max_over_ranks(time.perf_counter() - t0, dev)
    return world * E * n_e2e / e2e_s


DUMP_OBS_ENVS = 512  # observations of at most this many envs: 512 x 23,040 values x 4 B = 47 MB of float32


def dump_outputs(out_dir, obs, reward, done, info_sum):
    """--dump-outputs: what the caller of the timed path (rank 0's E envs) holds after its last step, as DIR/<name>.npy --
    obs.npy      float32 [n, 72, 80, 4]  the step's observations of n = min(E, DUMP_OBS_ENVS) envs: all of them, or for
                                         larger batches the envs numpy.random.default_rng(0).choice(E, n, replace=False)
                                         picks, in ascending order;
    reward.npy   float64 [E]             the step's rewards;
    done.npy     float32 [E]             the step's done flags;
    info_sum.npy float64 [72]            the episode-info sums of the last reduction.
    The actions come from a seeded generator and every env starts from the same state, so the same arguments give the same
    inputs on every run and every build."""
    import numpy as np
    import torch

    from pokegym_b200 import _capi

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    E = obs.shape[0]
    ids = np.sort(np.random.default_rng(0).choice(E, DUMP_OBS_ENVS, replace=False)) if E > DUMP_OBS_ENVS else np.arange(E)
    sample = obs[torch.from_numpy(ids).to(obs.device)].cpu().numpy()
    np.save(out / "obs.npy", sample.reshape(len(ids), _capi.OBS_H, _capi.OBS_W, _capi.OBS_C).astype(np.float32))
    np.save(out / "reward.npy", reward.cpu().numpy().astype(np.float64))
    np.save(out / "done.npy", done.cpu().numpy().astype(np.float32))
    np.save(out / "info_sum.npy", info_sum.cpu().numpy().astype(np.float64))


def run_leg(lib, rom, E, steps, warmup, preroll, dev, device_id, seed=7, state_path=None, mixed=False, lanes=None, e2e_steps=0):
    """One single-GPU workload: E envs, device-resident actions, obs into a 4-deep device ring.  CUDA-event timed."""
    import torch

    from pokegym_b200 import _capi

    h = _capi.Handle(lib, E, rom, device_id=device_id)
    if lanes:
        h.set_lanes_per_warp(lanes)
    start_envs(h, state_path, E, mixed)
    ring = torch.zeros((4, E, _capi.OBS_BYTES), dtype=torch.uint8, device=dev)
    rew = torch.zeros(E, dtype=torch.float64, device=dev)
    done = torch.zeros(E, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    total = preroll + warmup + steps
    actions = torch.randint(0, 8, (min(total, 512), E), generator=gen, device=dev, dtype=torch.uint8)
    h.reset(ring[0])
    for i in range(preroll + warmup):
        h.step(actions[i % 512], ring[i % 4], rew, done)
    torch.cuda.synchronize()
    c0, k0 = h.counters(), h.kernel_time_total(0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(preroll + warmup, total):
        h.step(actions[i % 512], ring[i % 4], rew, done)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    c1, k1 = h.counters(), h.kernel_time_total(0)
    rec = {"envs_per_gpu": E, "value": E * steps / (ms / 1000.0), "unit": "env-steps/s", "steps": steps, "warmup": warmup, "preroll": preroll,
           "ms_per_step": ms / steps, "kernel_ms": (k1[0] - k0[0]) / max(1, k1[1] - k0[1]),
           "emulated_instr_per_s": (c1.instructions - c0.instructions) / (ms / 1000.0),
           "emulated_instr_per_env_step": (c1.instructions - c0.instructions) / (E * steps), "faults": int(c1.faults), "lanes_per_warp": h.lanes_per_warp()}
    if e2e_steps:
        del ring
        torch.cuda.empty_cache()
        v = e2e_host_loop(h, E, e2e_steps)
        rec["e2e"] = {"value": v, "unit": "env-steps/s", "steps": e2e_steps, "h2d_bytes_per_step": E, "d2h_bytes_per_step": E * (_capi.OBS_BYTES + 8 + 1),
                      "share_of_value": v / rec["value"], "api": "gbenv_submit_host / gbenv_fetch_host (pinned host buffers, two steps in flight)"}
        ring = None
    h.close()
    del ring
    torch.cuda.empty_cache()
    return rec


LEGS = {
    # name: (rom, envs, steps, warmup, preroll, mixed states)
    "main_4096": ("pokelike", 4096, 40, 5, 150, False),  # the headline workload as a leg (tools/gpu_exp2.sh: lanes sweeps)
    "envs_32768": ("pokelike", 32768, 20, 5, 100, False),
    "busy_4096": ("busy", 4096, 12, 3, 30, False),
    "timer_4096": ("pokelike_timer", 4096, 20, 5, 60, False),
    "divergent_4096": ("pokelike", 4096, 40, 5, 100, True),
    "divergent_32768": ("pokelike", 32768, 16, 4, 60, True),
    "n72": ("pokelike", 72, 100, 10, 100, False),
    "n1": ("pokelike", 1, 100, 10, 50, False),
}


def run_single_config(args):
    """BASELINE.json config 1 with the protocol of the reference's test.py:16-29 -- one pokegym.Environment, 1,000 warm-up
    steps, 10,000 x step(0) -- through the drop-in facade (pokegym_b200.Environment, a batch of one on the GPU), beside ONE
    host thread of the oracle port."""
    import torch

    from pokegym_b200 import Environment

    rom = build_rom(args.rom)
    warm, steps = (1000, 10000) if args.steps is None else (max(args.warmup, 3), args.steps)
    env = Environment(rom, state_path=args.state)
    env.reset()
    for _ in range(warm):
        env.step(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        env.step(0)
    dt = time.perf_counter() - t0
    env.close()
    v, cores, sample = oracle_run(rom, min(args.cpu_baseline_seconds, 10.0), n_envs=1, state_path=args.state)
    line = {"metric": "env_steps_per_s", "value": steps / dt, "unit": "env-steps/s", "n_gpus": 1, "steps": steps, "warmup": warm,
            "ms_per_step": 1000.0 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "BASELINE.json config 1: single pokegym_b200.Environment, step(0), protocol of the reference's test.py:16-29",
                       "rom": args.rom, "envs_per_gpu": 1,
                       "note": "one env cannot fill a GPU: a single interpreter thread is latency bound; below ~300 envs the CPU port is faster"},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": 1, "kind": "port", "sample": sample},
            "e2e": {"value": steps / dt, "unit": "env-steps/s", "h2d_bytes_per_step": 1, "d2h_bytes_per_step": 23040 + 9, "api": "pokegym_b200.Environment.step"},
            "gpu_launches": 3 * steps}
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    import numpy as np  # noqa: F401
    import torch
    import torch.distributed as dist

    import __graft_entry__ as g
    from pokegym_b200 import _capi
    from pokegym_b200.dist import all_reduce_info, max_over_ranks
    from pokegym_b200.groups import EnvGroups

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.config == "single":
        if library(g.build_cuda) != _capi.DEFAULT_LIB:  # pokegym_b200.Environment loads the in-tree library
            raise SystemExit(f"{_capi.DEFAULT_LIB} is older than its sources: run build() before --config single")
        run_single_config(args)
        return
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # GBENV_LIB: another build of the kernel library, for A/B runs while tuning (tools/gpu_variants.sh)
    lib = _capi.GbEnvLib(os.environ.get("GBENV_LIB") or library(g.build_cuda))
    if args.only_leg:
        if args.only_leg.startswith("custom:"):  # custom:rom,envs,steps,warmup,preroll,mixed  (tuning sweeps)
            f = args.only_leg[7:].split(",")
            LEGS[args.only_leg] = (f[0], int(f[1]), int(f[2]), int(f[3]), int(f[4]), bool(int(f[5])))
        rom_name, E, steps, warmup, preroll, mixed = LEGS[args.only_leg]
        rec = run_leg(lib, build_rom(rom_name), E, steps, warmup, preroll, dev, local_rank, mixed=mixed, e2e_steps=8 if args.only_leg == "envs_32768" else 0)
        rec["leg"] = args.only_leg
        print(json.dumps(rec))
        return
    E, K, W = args.envs_per_gpu, args.steps, max(args.warmup, 3)
    rom = build_rom(args.rom)
    props = torch.cuda.get_device_properties(dev)
    # Env groups (pokegym_b200.EnvGroups): while every env has a warp of its own (the emulation kernel is then bound by
    # instruction issue) the batch steps as two groups on two streams, so that the tail of one group's launch -- its few
    # slowest envs -- is filled by the other group; bigger batches are latency bound and gain nothing from it.
    G = args.groups if args.groups > 0 else (2 if E <= props.multi_processor_count * 32 and E % 64 == 0 else 1)
    h = EnvGroups(lib, E, rom, n_groups=G, device_id=local_rank)
    h.for_each(lambda hh, g, st: start_envs(hh, args.state, E // G))  # every env starts from the same state and diverges through its actions
    rollout = torch.zeros((ROLLOUT_T, E, _capi.OBS_BYTES), dtype=torch.uint8, device=dev)
    reward = torch.zeros((ROLLOUT_T, E), dtype=torch.float64, device=dev)
    done = torch.zeros((ROLLOUT_T, E), dtype=torch.uint8, device=dev)
    info_sum = torch.zeros(_capi.INFO_SCALARS, dtype=torch.float64, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    n_act = 512
    actions = torch.randint(0, 8, (n_act, E), generator=gen, device=dev, dtype=torch.uint8)
    torch.cuda.synchronize()
    h.reset(rollout[0])
    reduces = 0

    def reduce_info():  # episode-info scalars summed over envs, then over ranks (the path's only collective)
        nonlocal reduces
        h.reduce_info(info_sum)  # joins the groups: the rollout is complete here
        all_reduce_info(info_sum)  # NCCL sum over ranks (a no-op for one rank)
        reduces += 1

    def step(i):
        t = i % ROLLOUT_T
        h.step(actions[i % n_act], rollout[t], reward[t], done[t])
        if t == ROLLOUT_T - 1:  # once per rollout
            reduce_info()

    for i in range(args.preroll + W):
        step(i)
    h.join()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    c0 = h.counters()
    k0 = h.kernel_time_total(0)
    k1 = h.kernel_time_total(1)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    reduces = 0
    ev0.record()
    for i in range(args.preroll + W, args.preroll + W + K):
        step(i)
    if reduces == 0:  # a short run ends inside a rollout: the reduction still belongs to the timed region
        reduce_info()
    h.join()  # the timed region ends when every group has finished its last step
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    c1 = h.counters()
    k0b = h.kernel_time_total(0)
    k1b = h.kernel_time_total(1)
    if world > 1:
        dist.barrier()
    ms = max_over_ranks(ms, dev)
    value = world * E * K / (ms / 1000.0)
    if args.dump_outputs and rank == 0:
        t = (args.preroll + W + K - 1) % ROLLOUT_T  # rollout slot of the last timed step
        dump_outputs(args.dump_outputs, rollout[t], reward[t], done[t], info_sum)

    # ---- end to end through the host-buffer entry points (pinned memory, copies inside the timed region).  Double
    # buffered: step t+1 is submitted before the results of step t are fetched, so the 94 MB D2H of the observations
    # overlaps the next emulation kernel -- what a vectoriser that keeps two rollout slots in flight does.
    n_e2e = max(3, min(args.e2e_steps, K))
    e2e_value = e2e_host_loop(h.handles, E, n_e2e, world, dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (k_run_frames), from CUDA events on its launching stream
    run_ms = (k0b[0] - k0[0]) / max(1, k0b[1] - k0[1])
    wrap_ms = (k1b[0] - k1[0]) / max(1, k1b[1] - k1[1])
    peak, peak_src = measured_peak()
    # one launch steps one group; the G launches of a step run side by side (each lasts run_ms, the step barely longer), so the
    # rate the machine sustains is the bytes of all G over that duration
    achieved = ALGO_BYTES_PER_ENV_STEP * (E // G) * G / (run_ms / 1000.0) / 1e9
    counters = recorded_counters()
    instr = c1.instructions - c0.instructions
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    line = {
        "metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_name(args), "envs_per_gpu": E, "act_freq": 24, "rom": args.rom, "parallelism": f"env-sharded x{world}",
                   "env_groups": G, "env_groups_note": (f"{G} groups of {E // G} envs step on {G} CUDA streams (pokegym_b200.EnvGroups)"
                                                        + ("; the single-group figure is legs.main_4096" if world == 1 else "") if G > 1 else "one group"),
                   "preroll_steps": args.preroll, "info_allreduces_in_timed_region": reduces,
                   "l2_policy": f"working set {E * (16896 + 5760 + 23040 + 1152) / 1e6:.0f} MB of env state + obs per GPU exceeds the 126 MB L2; no explicit flush"},
        "frames_per_s": 24 * value,
        "emulated_instr_per_s": instr / (ms / 1000.0) * world,
        "roofline": {"bound": "hbm", "kernel": "k_run_frames", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": (counters or {}).get("dram_bytes_per_launch"), "peak_source": peak_src,
                     "kernel_ms": run_ms, "launches_per_step": G, "concurrent_launches": G, "envs_per_launch": E // G,
                     "kernel_share_of_step": run_ms / (ms / K) if G == 1 else None, "wrap_kernels_ms": wrap_ms,
                     "algorithmic_bytes_per_launch": ALGO_BYTES_PER_ENV_STEP * (E // G),
                     "note": "the HBM figure is the prescribed one; the kernel is an interpreter and is bounded by instruction issue, see `issue`"
                             + (f"; the {G} launches of a step (one per env group) run concurrently: kernel_ms is the event-timed duration of one of them while the "
                                f"others run beside it, and `achieved` counts the algorithmic bytes of all {G} over that duration" if G > 1 else "")},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": E, "d2h_bytes_per_step": E * (_capi.OBS_BYTES + 8 + 1),
                "steps": n_e2e, "api": "gbenv_submit_host / gbenv_fetch_host (pinned host buffers, two steps in flight)"},
        "gpu_launches": int(c1.kernel_launches - c0.kernel_launches),
        "clocks": clocks,
        "faults": int(c1.faults),
    }
    if counters and counters.get("envs_per_launch") == E // G:
        line["issue"] = issue_record(counters, run_ms / G, sm_mhz, props.multi_processor_count)  # G launches share the machine
    want = [] if args.legs == "none" else ([x for x in LEGS if G > 1 or x != "main_4096"] if args.legs == "all" else [x for x in args.legs.split(",") if x in LEGS])
    if world == 1 and want:
        h.close()
        del rollout
        torch.cuda.empty_cache()
        line["legs"] = {}
        for name in want:
            rom_name, E2, steps, warmup, preroll, mixed = LEGS[name]
            try:
                rec = run_leg(lib, rom if rom_name == args.rom else build_rom(rom_name), E2, steps, warmup, preroll, dev, local_rank, mixed=mixed,
                              e2e_steps=8 if name == "envs_32768" else 0)
                rec["workload"] = f"{rom_name} ROM" + (", env i reset from reference save-state i mod 40 (BASELINE.json config 5)" if mixed else "")
                lc = recorded_counters(f"r2_{name}_counters.json")
                if lc and lc.get("envs_per_launch") == E2:
                    rec["issue"] = issue_record(lc, rec["kernel_ms"], sm_mhz, props.multi_processor_count)
                line["legs"][name] = rec
            except Exception as e:
                line["legs"][name] = {"error": str(e)}
        if args.also_envs < 0:
            args.also_envs = props.multi_processor_count * 20 * 32  # 94,720 on a 148-SM B200: every warp slot of a 10-block SM full
        if args.also_envs and args.also_envs != E:
            # throughput keeps growing with the number of resident envs: the full-wave point next to the headline
            try:
                line["large_batch"] = run_leg(lib, rom, args.also_envs, args.also_steps, 3, 30, dev, local_rank)
            except Exception as e:
                line["large_batch"] = {"error": str(e)}
    try:
        v, cores, sample = oracle_run(rom, args.cpu_baseline_seconds, state_path=args.state)
        line["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample}
        if world == 1 and "legs" in line and "divergent_4096" in line["legs"]:
            v2, _, s2 = oracle_run(rom, min(args.cpu_baseline_seconds, 6.0), mixed=True)
            line["legs"]["divergent_4096"]["cpu_baseline"] = {"value": v2, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": s2}
    except Exception as e:  # the baseline is reported, never required for the GPU number
        line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    tb = tier_b_record()
    if tb:
        line["cpu_baseline_tier_b"] = tb
    line["pyboy_baseline"] = "not run (PyBoy / Pokemon Red ROM missing): cpu_baseline is the oracle port, tier B the reference wrapper over it"
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
