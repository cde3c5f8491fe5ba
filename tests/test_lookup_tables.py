"""The lookup tables of the single-lane fast body (gb_cpu.cuh) against the compare chains and flag arithmetic they replace.

Compiles the device headers on the host (GB_HOSTSIM, like tests/hostsim) into a small program that walks all 65,536
addresses and all 512 INC / DEC inputs and prints every disagreement.
"""
import shutil
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent

PROGRAM = r"""
#define GB_HOSTSIM 1
#include "pokegym_b200/csrc/gb_hd.h"
#include "pokegym_b200/csrc/gb_kernels.cuh"
#include <stdio.h>

int main() {
    int bad = 0;
    for (uint32_t a = 0; a < 0x10000u; a++) {
        // the compare chains of the single-lane body before the tables: store target, read, deferred-PPU test
        uint32_t want_wt = FAST_WR_NONE;
        if (a - 0xC000u < 0x3E00u) want_wt = mem_offset(MEM_WRAM + (a & 0x1FFF));
        else if (a - 0xFF80u < 0x7Fu || a - 0xFE00u < 0x100u) want_wt = mem_offset(MEM_HI + (a - 0xFE00));
        else if (a - 0x8000u < 0x2000u) want_wt = mem_offset(MEM_VRAM + (a - 0x8000));
        else if (a - 0x2000u < 0x2000u) want_wt = FAST_WR_BANK;
        else if (a - 0xFF10u < 0x30u) want_wt = FAST_WR_DROP;
        else if (a == 0xFF00u) want_wt = FAST_WR_P1;
        uint32_t plain_off;
        const bool plain = fast_plain_offset(a, plain_off);  // the lock-step build's reads: plain RAM
        const bool want_rd = a >= 0x8000u && (plain || a - 0xFF00u < 4u);
        const bool want_defer = a - 0x8000u < 0x2000u || a - 0xFE00u < 0x100u;
        uint32_t e;
        const uint32_t wt = fast_store_target_map(a, e);
        const bool rd = (e & GB_MAP_RD) != 0;
        if (wt != want_wt || (a >= 0x8000u && rd != want_rd) || (rd && gb_map_offset(a, e) != (plain ? plain_off : mem_offset(MEM_HI + (a - 0xFE00)))) ||
            ((e & GB_MAP_DEFER) != 0) != want_defer) {
            if (bad++ < 10) printf("address %04x: entry %08x store %08x (want %08x) read %d (want %d)\n", a, e, wt, want_wt, rd, want_rd);
        }
    }
    for (uint32_t dec = 0; dec < 2; dec++) {
        for (uint32_t b = 0; b < 256; b++) {
            for (uint32_t f = 0; f < 0x100u; f += 0x10u) {
                const uint32_t op = dec ? 0xFFu : 1u, ex = dec ? 0x60u : 0u, sum = b + op, res = sum & 0xFF;
                const uint32_t want = res | (((f & FLAG_C) | ((((b ^ op ^ sum) & 0x10) << 1) ^ ex) | (res == 0 ? FLAG_Z : 0)) << 8);
                const uint32_t dx = 4u | (op << 8) | (ex << 16), hlaf = f << 24;
                const uint32_t got = c_incdec[256 + (int)gb_prmt(b, dx, 0xDDD0u)] | ((hlaf >> 16) & (FLAG_C << 8));
                if (got != want && bad++ < 20) printf("%s %02x F %02x: %04x want %04x\n", dec ? "DEC" : "INC", b, f, got, want);
            }
        }
    }
    printf("%d mismatches\n", bad);
    return bad != 0;
}
"""


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_memory_map_and_incdec_tables_match_the_arithmetic(tmp_path):
    src = tmp_path / "tables.cpp"
    src.write_text(PROGRAM)
    exe = tmp_path / "tables"
    subprocess.run(["g++", "-O1", "-std=c++17", "-Wno-unknown-pragmas", "-I", str(ROOT), "-o", str(exe), str(src)], check=True)
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0, run.stdout
