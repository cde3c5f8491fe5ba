"""gb_classes.inc is generated (tools/gen_classes.sh) from the per-opcode base table and the class mix of the benchmark
workloads (tools/class_counts.txt): the committed file must be what the generator makes of the committed inputs, so that
the class order and the single-lane dispatch tree have one source."""
import shutil
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_gb_classes_inc_matches_generator(tmp_path):
    exe = tmp_path / "gen_classes"
    subprocess.run(["g++", "-std=c++17", "-I", str(ROOT / "pokegym_b200" / "csrc"), "-o", str(exe), str(ROOT / "tools" / "gen_classes.cpp")], check=True)
    out = subprocess.run([str(exe), str(ROOT / "tools" / "class_counts.txt")], check=True, capture_output=True, text=True).stdout
    assert out == (ROOT / "pokegym_b200" / "csrc" / "gb_classes.inc").read_text()
    assert "GB_CLS_DISPATCH" in out
