#!/bin/bash
# Regenerates pokegym_b200/csrc/gb_classes.inc from the per-opcode base table of gb_predecode.h and the class mix in
# tools/class_counts.txt (run after changing pd_build_base; refresh the mix with tools/class_mix.py).
set -e
cd "$(dirname "$0")/.."
tmp=$(mktemp -d)
trap 'rm -rf "$tmp"' EXIT
g++ -std=c++17 -I pokegym_b200/csrc -o "$tmp/gen_classes" tools/gen_classes.cpp
"$tmp/gen_classes" tools/class_counts.txt > "$tmp/gb_classes.inc"
mv "$tmp/gb_classes.inc" pokegym_b200/csrc/gb_classes.inc
grep GB_CLS_COUNT pokegym_b200/csrc/gb_classes.inc
