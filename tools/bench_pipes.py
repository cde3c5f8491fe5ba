#!/usr/bin/env python
"""Pipe map of the GPU: warp instructions per cycle per SM of each SASS operation the interpreter uses (tools/bench_pipes.cu).

    python tools/bench_pipes.py [--out profiles/pipes_b200.json]

Compiles bench_pipes.cu for sm_100a into a temporary directory, checks in its SASS that every stream consists of the
operation it is named after (the record keeps the opcode counts of each kernel), runs it and writes one JSON record with
the card's name and power limit.  An operation shares the integer ALU pipe with LOP3 when the 1:1 mix of the two runs no
faster than the slower of them alone (on two pipes it would run at twice that); `alu_pipe` lists those.
tools/alu_cost.py reads the record.
"""
from __future__ import annotations

import argparse
import collections
import json
import re
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
SRC = ROOT / "tools" / "bench_pipes.cu"
# stream -> SASS opcode (prefix) it must consist of; LEA and the plain add are issued by ptxas as a mix of two opcodes
EXPECT = {
    "LOP3": ["LOP3"], "SHF": ["SHF"], "PRMT": ["PRMT"], "IADD3": ["IADD3"], "SEL": ["SEL"], "ISETP": ["ISETP"],
    "LEA": ["LEA", "IMAD"], "IMAD": ["IMAD"], "IMAD_IADD": ["IMAD.IADD", "IADD3"], "LDC": ["LDC"], "LDS": ["LDS"],
    "MIX_SHF": ["SHF"], "MIX_PRMT": ["PRMT"], "MIX_IADD3": ["IADD3"], "MIX_SEL": ["SEL"], "MIX_ISETP": ["ISETP"],
    "MIX_LEA": ["IMAD"], "MIX_VIADD": ["VIADD"], "MIX_IMAD": ["IMAD"], "MIX_IMAD_SHL": ["IMAD.SHL"],
    "MIX_IMAD_IADD": ["IMAD.IADD"], "MIX_LDC": ["LDC"], "MIX_LDS": ["LDS"],
}
STEPS_PER_ITER = 16 * 8  # UNROLL x CHAINS of bench_pipes.cu


def sass_counts(binary: Path) -> dict:
    out = subprocess.run(["cuobjdump", "-sass", str(binary)], check=True, capture_output=True, text=True).stdout
    cur, counts = None, {}
    for line in out.splitlines():
        m = re.search(r"Function : _Z\d+k_(\w+?)jPjPx", line)
        if m:
            cur = m.group(1)
            counts[cur] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_.]+)", line)
        if m and cur:
            counts[cur][m.group(1)] += 1
    return counts


def check_streams(counts: dict) -> dict:
    """opcode counts of the stream operation(s) per kernel; raises when a stream lost its operation"""
    kept = {}
    for name, ops in EXPECT.items():
        c = counts[name]
        found = {op: n for op, n in c.items() if any(op.startswith(p) for p in ops)}
        if sum(found.values()) < STEPS_PER_ITER:
            raise SystemExit(f"stream {name}: expected {ops} in its SASS, found {c.most_common(4)}")
        kept[name] = found
    return kept


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON record to write (default: print only)")
    args = ap.parse_args()
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    with tempfile.TemporaryDirectory(prefix="bench-pipes-") as tmp:
        exe = Path(tmp) / "bench_pipes"
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-diag-suppress", "550",
                        "-o", str(exe), str(SRC)], check=True)
        sass = check_streams(sass_counts(exe))
        run = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    rates, device = {}, None
    for line in run.splitlines():
        if line.startswith("device "):
            device = line[len("device "):]
        else:
            k, v = line.split()
            rates[k] = float(v)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lop3 = rates["LOP3"]
    alone = {k: v for k, v in rates.items() if not k.startswith("MIX_")}
    mixes = {k[4:]: v for k, v in rates.items() if k.startswith("MIX_")}
    # two pipes run a 1:1 mix at twice the slower rate, one shared pipe at its own rate; the table loads are latency-bound
    # streams, not a pipe test, and ptxas issues the LEA stream as half LEA, half IMAD, so neither can be classified this way
    alu = ["LOP3"] + sorted(op for op, r in mixes.items()
                            if op not in ("LDC", "LDS", "LEA") and r < 1.25 * min(lop3, alone.get(op, r)))
    rec = {
        "what": "warp instructions per cycle per SM of long independent streams of one SASS operation (tools/bench_pipes.cu); "
                "MIX_x: x and LOP3 1:1; 4.0 = one per cycle on each of the SM's four schedulers",
        "device": device, "nvidia_smi": smi[0] if smi else None,
        "rates": alone, "mix_with_lop3": mixes, "alu_pipe": alu,
        "assumed_alu_pipe": {"ops": ["LEA", "PLOP3"], "why": "no stream of its own (ptxas mixes LEA with IMAD; PLOP3 only "
                             "combines predicates); counted at the LOP3 rate"},
        "sass": sass,
    }
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    sys.exit(main())
