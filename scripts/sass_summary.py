#!/usr/bin/env python
"""SASS facts of the hot kernels (what DESIGN.md quotes), from the built objects: instruction count, the mnemonics that prove
the mechanism (UBLKCP = cp.async.bulk, SYNCS = mbarrier, LDGSTS = cp.async, UCGABAR = cluster barrier, IMAD.WIDE = the
Montgomery chains, 128-bit loads / stores), registers and shared memory.  usage: python scripts/sass_summary.py > profiles/rNN_sass_summary.txt"""
import os
import re
import subprocess
import sys
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "zkinterface-ir_b200", "build")
# Lj0 / Lj1: the generic Montgomery product / the one for moduli whose low 64 bits are 2^64 - 2^32 + 1 (FieldParams::mul_form)
KERNELS = [("kernels.cu.o", "k_level_tmaILi8ELj0"), ("kernels.cu.o", "k_level_tmaILi8ELj1"), ("kernels.cu.o", "k_level_pipeILi8ELi1ELj0"),
           ("kernels.cu.o", "k_level_pipeILi8ELi1ELj1"), ("kernels.cu.o", "k_arith_groupsILi8ELj0"), ("kernels.cu.o", "k_arith_groupsILi8ELj1"),
           ("kernels.cu.o", "k_level_pipeILi2ELi2"),
           ("kernels.cu.o", "k_levels_coopILi8ELb0"), ("kernels.cu.o", "k_levels_coopILi2ELb1"), ("kernels.cu.o", "k_levels_flowILi2"),
           ("kernels.cu.o", "k_levels_flow_wideILi8"), ("kernels.cu.o", "k_bool_levelILi4"), ("kernels.cu.o", "k_bool_groupsILi1"),
           ("kernels.cu.o", "k_bool_groupsILi4"), ("kernels.cu.o", "k_load_inputsILi8"), ("r1cs.cu.o", "k_r1cs_checkILi8"),
           ("r1cs.cu.o", "k_r1cs_checkILi4")]
WATCH = ["IMAD.WIDE", "IMAD", "IADD3", "LOP3", "LDG.E.128", "LDG", "STG.E.128", "STG", "LDS", "STS", "LDGSTS", "UBLKCP", "SYNCS", "UCGABAR",
         "BAR.SYNC", "LD.E", "ST.E", "NANOSLEEP", "ATOMG", "REDUX", "VOTE", "LDC", "BRA"]


def functions(obj):
    txt = subprocess.run(["cuobjdump", "-sass", os.path.join(BUILD, obj)], capture_output=True, text=True).stdout
    cur, out = None, {}
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m and cur:
            out[cur].append(m.group(1))
    return out


def resources(obj):
    txt = subprocess.run(["cuobjdump", "-res-usage", os.path.join(BUILD, obj)], capture_output=True, text=True).stdout
    out, cur = {}, None
    for line in txt.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            cur = m.group(1)
        m = re.search(r"REG:(\d+).*SHARED:(\d+)", line)
        if m and cur:
            out[cur] = (int(m.group(1)), int(m.group(2)))
    return out


def main():
    cache, res = {}, {}
    print("kernel | instructions | registers | static smem | " + " | ".join(WATCH))
    for obj, key in KERNELS:
        if obj not in cache:
            cache[obj], res[obj] = functions(obj), resources(obj)
        names = [n for n in cache[obj] if key in n]
        if not names:
            print(f"{key} | (not found)")
            continue
        n = names[0]
        ins = cache[obj][n]
        cnt = Counter()
        for i in ins:
            for w in WATCH:
                if i == w or i.startswith(w + ".") or i.startswith(w + "_"):
                    cnt[w] += 1
        reg, sh = res[obj].get(n, (0, 0))
        print(f"{key} | {len(ins)} | {reg} | {sh} | " + " | ".join(str(cnt[w]) for w in WATCH))


if __name__ == "__main__":
    main()
