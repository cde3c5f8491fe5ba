#!/usr/bin/env python
"""Static cost model of the single-lane interpreter loop: issue slots and integer-ALU-pipe cycles per emulated instruction.

    python tools/alu_cost.py LIB_OR_SASS [--pipes profiles/pipes_b200.json] [--share 0.95] [-v]

Reads the SASS of k_run_frames_1 (`cuobjdump -sass` of a built libgbenv.so, or a saved dump) and, for each class of the
class-dispatched fast loop that makes up the first `share` of tools/class_counts.txt, walks the common path of one
emulated instruction: loop head -> control-word fetch (ROM code) -> the dispatch tree (its tests on the class id are
evaluated for that class) -> the class body -> loop tail -> back edge.  Inside the body the path is the shortest one (in
SASS instructions) back to the loop head that stays inside the loop, which excludes declines (they leave for the slow tick)
and the deadline exit; a class that reads memory must pass a byte load from the env's RAM (not a ROM load), a class that
stores one must pass a byte store.  Conditional jumps, RET and CALL take whichever of taken / not taken is shorter.
Issue slots count every SASS instruction on the path; ALU-pipe cycles count the instructions of the pipe map's `alu_pipe`
operations at 4 / (their measured warp instructions per cycle per SM), i.e. cycles of one scheduler's ALU pipe.  Both
are printed per class and as the average weighted by the class counts.
"""
from __future__ import annotations

import argparse
import json
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
KERNEL = "_Z14k_run_frames_19RunParams"
# without a pipe map: the operations of the integer ALU pipe at half rate (2 warp instructions per cycle per SM)
DEFAULT_ALU = {"LOP3": 2.0, "ISETP": 2.0, "SHF": 2.0, "PRMT": 2.0, "IADD3": 2.0, "SEL": 2.0, "LEA": 2.0, "PLOP3": 2.0}
# pipe-map stream name -> SASS opcode prefix it measures
STREAM_OP = {"LOP3": "LOP3", "SHF": "SHF", "PRMT": "PRMT", "IADD3": "IADD3", "SEL": "SEL", "ISETP": "ISETP", "LEA": "LEA",
             "VIADD": "VIADD", "IMAD": "IMAD", "IMAD_SHL": "IMAD.SHL", "IMAD_IADD": "IMAD.IADD", "LDC": "LDC", "LDS": "LDS"}
PDF_RD, PDF_WR = 0x0020, 0x0200


def load_sass(src: str) -> list:
    text = Path(src).read_text() if src.endswith(".sass") or src.endswith(".txt") else subprocess.run(
        ["cuobjdump", "-sass", "-fun", KERNEL, src], check=True, capture_output=True, text=True).stdout
    ins, on = [], False
    for line in text.splitlines():
        if "Function :" in line:
            on = KERNEL in line
            continue
        m = re.match(r"\s+/\*([0-9a-f]+)\*/\s+(@!?U?P[T0-9]+\s+)?([A-Z0-9_.]+)\s*([^;]*);", line)
        if on and m:
            ins.append({"addr": int(m.group(1), 16), "pred": (m.group(2) or "").strip(), "op": m.group(3), "args": m.group(4).strip()})
    if not ins:
        raise SystemExit(f"no SASS of {KERNEL} in {src}")
    return ins


def classes() -> tuple[dict, dict]:
    """class id -> (handler, flags) from gb_classes.inc; (handler, flags) -> count from tools/class_counts.txt"""
    inc = (ROOT / "pokegym_b200" / "csrc" / "gb_classes.inc").read_text()
    ids = {int(i): (int(h), int(f, 16)) for i, h, f in re.findall(r"^GB_CLS\((\d+), (\d+), (0x[0-9a-f]+)u\)", inc, re.M)}
    counts = {}
    for line in (ROOT / "tools" / "class_counts.txt").read_text().splitlines():
        if line.startswith("#") or not line.strip():
            continue
        h, f, n = line.split()
        counts[(int(h), int(f, 16))] = int(n)
    return ids, counts


def branch_target(i: dict):
    m = re.search(r"0x([0-9a-f]+)\s*$", i["args"])
    return int(m.group(1), 16) if m else None


def cmp_eval(cmp: str, a: int, b: int) -> bool:
    return {"EQ": a == b, "NE": a != b, "LT": a < b, "LE": a <= b, "GT": a > b, "GE": a >= b}[cmp]


class Loop:
    def __init__(self, ins: list):
        self.ins = ins
        self.at = {x["addr"]: k for k, x in enumerate(ins)}
        # the class dispatch: class id = control word w >> 24 (SHF.R.U32.HI Rc, RZ, 0x18, Rw), then compares of Rc with constants;
        # the class loop's control-word load is the LDG.E.128 whose fall-through jumps there
        self.head = self.dispatch = self.creg = None
        for k, x in enumerate(ins):
            if x["op"].startswith("LDG.E.128") and ins[k + 1]["op"] == "BRA" and not ins[k + 1]["pred"]:
                d = self.at[branch_target(ins[k + 1])]
                m = re.match(r"(R\d+), RZ, 0x18, R(\d+)", ins[d]["args"])
                w = int(re.match(r"R(\d+)", x["args"]).group(1)) + 3
                if ins[d]["op"] == "SHF.R.U32.HI" and m and int(m.group(2)) == w and ins[d + 1]["op"].startswith("ISETP"):
                    self.dispatch, self.creg, ldg = d, m.group(1), x["addr"]
        if self.dispatch is None:
            raise SystemExit("class dispatch not found")
        backs = [(branch_target(x), x["addr"]) for x in ins if x["op"] == "BRA" and not x["pred"] and x["addr"] > ldg
                 and branch_target(x) is not None and branch_target(x) <= ldg]
        self.head = self.at[max(t for t, _ in backs)]
        self.end = max(s for t, s in backs if t == self.ins[self.head]["addr"])

    def pred_def(self, k: int, p: str):
        """the instruction of k's basic block that last wrote predicate p before k"""
        targets = {branch_target(x) for x in self.ins if x["op"] == "BRA"}
        j = k - 1
        while j >= 0 and self.ins[j + 1]["addr"] not in targets:
            a = self.ins[j]["args"]
            if re.match(rf"{p}\b", a) and not self.ins[j]["pred"]:
                return self.ins[j]
            if self.ins[j]["op"] == "BRA":
                return None
            j -= 1
        return None

    def static_branch(self, k: int, cls: int):
        """True / False when branch k tests the class id against a constant (taken or not for class cls), else None"""
        x = self.ins[k]
        m = re.match(r"@(!?)(P\d)", x["pred"])
        if not m or "," in x["args"]:
            return None
        d = self.pred_def(k, m.group(2))
        if d is None or not d["op"].startswith("ISETP"):
            return None
        mm = re.match(r"ISETP\.(\w\w)(\.U32)?\.AND$", d["op"])
        aa = [s.strip() for s in d["args"].split(",")]
        if not mm or len(aa) != 5 or aa[1] != "PT" or aa[4] != "PT" or aa[2] != self.creg:
            return None
        b = 0 if aa[3] == "RZ" else int(aa[3], 16) if aa[3].startswith("0x") else None
        if b is None:
            return None
        v = cmp_eval(mm.group(1), cls, b)
        return v != (m.group(1) == "!")

    def succ(self, k: int, cls: int):
        x = self.ins[k]
        if x["op"] in ("EXIT", "RET.REL.NODEC", "RET.ABS.NODEC") or x["op"].startswith("RET"):
            return []
        if x["op"] == "BRA":
            t = self.at.get(branch_target(x))
            if not x["pred"] or x["pred"] == "@PT":
                return [t]
            s = self.static_branch(k, cls)
            if s is True:
                return [t]
            if s is False:
                return [k + 1]
            return [t, k + 1]
        return [k + 1]

    def path(self, cls: int, need_load: bool, need_store: bool):
        """shortest path head -> head through the body of class cls (list of instruction indices)"""
        lo, hi = self.ins[self.head]["addr"], self.end

        def marks(k):
            x = self.ins[k]
            ld = bool(re.match(r"LDG?\.E\.U8$", x["op"]) or x["op"] in ("LD.E.U8", "LDG.E.U8"))
            st = x["op"] in ("ST.E.U8", "STG.E.U8")
            return ld, st

        def flags(k, hl, hs):
            ld, st = marks(k)
            return hl or ld, hs or st

        # breadth-first over (instruction, load seen, store seen): every instruction costs one issue slot
        first = (self.head, *flags(self.head, not need_load, not need_store))
        queue, prev, qi = [first], {first: None}, 0
        while qi < len(queue):
            cur = queue[qi]
            qi += 1
            k, hl, hs = cur
            for n in self.succ(k, cls):
                if n is None or not (lo <= self.ins[n]["addr"] <= hi):
                    continue
                if n == self.head:
                    if hl and hs:
                        out = []
                        while cur is not None:
                            out.append(cur[0])
                            cur = prev[cur]
                        return out[::-1]
                    continue
                nxt = (n, *flags(n, hl, hs))
                if nxt not in prev:
                    prev[nxt] = cur
                    queue.append(nxt)
        return None


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("lib", help="libgbenv.so or a saved cuobjdump -sass dump (.sass / .txt)")
    ap.add_argument("--pipes", default=None, help="pipe map (tools/bench_pipes.py); default: LOP3 ISETP SHF PRMT IADD3 SEL LEA PLOP3 at half rate")
    ap.add_argument("--share", type=float, default=0.95)
    ap.add_argument("-v", action="store_true", help="print each class's path")
    args = ap.parse_args()
    if args.pipes:
        pm = json.loads(Path(args.pipes).read_text())
        alu = {STREAM_OP.get(s, s): pm["rates"].get(s) or pm["mix_with_lop3"].get(s) for s in pm["alu_pipe"]}
        alu = {op: r for op, r in alu.items() if r}
        alu.update({op: pm["rates"]["LOP3"] for op in pm.get("assumed_alu_pipe", {}).get("ops", [])})
    else:
        alu = dict(DEFAULT_ALU)
    ins = load_sass(args.lib)
    loop = Loop(ins)
    ids, counts = classes()
    by_hf = {hf: c for c, hf in ids.items()}
    total = sum(counts.values())
    rows, acc = [], 0
    for hf, n in sorted(counts.items(), key=lambda t: -t[1]):
        if acc >= args.share * total:
            break
        acc += n
        cls = by_hf[hf]
        p = loop.path(cls, bool(hf[1] & PDF_RD), bool(hf[1] & PDF_WR))
        if p is None:
            raise SystemExit(f"no path for class {cls} {hf}")
        alu_cyc = 0.0
        for k in p:
            op = ins[k]["op"]
            r = next((r for pre, r in sorted(alu.items(), key=lambda t: -len(t[0])) if op.startswith(pre)), None)
            alu_cyc += 4.0 / r if r else 0.0
        rows.append((cls, hf, n, len(p), alu_cyc))
        if args.v:
            print(f"class {cls} (handler {hf[0]}, flags {hf[1]:#06x}):")
            for k in p:
                print(f"    {ins[k]['addr']:05x} {ins[k]['pred']:>5} {ins[k]['op']} {ins[k]['args']}")
    w = sum(r[2] for r in rows)
    issue = sum(r[2] * r[3] for r in rows) / w
    alu_c = sum(r[2] * r[4] for r in rows) / w
    print(f"{'class':>5} {'handler':>7} {'flags':>7} {'share':>6} {'issue':>5} {'alu_cyc':>7}")
    for cls, hf, n, iss, ac in rows:
        print(f"{cls:5d} {hf[0]:7d} {hf[1]:#07x} {100 * n / total:5.1f}% {iss:5d} {ac:7.1f}")
    print(json.dumps({"classes_share": round(w / total, 4), "issue_per_instr": round(issue, 2), "alu_cycles_per_instr": round(alu_c, 2),
                      "alu_ops": sorted(alu)}))


if __name__ == "__main__":
    sys.exit(main())
