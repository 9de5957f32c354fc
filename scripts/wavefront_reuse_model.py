#!/usr/bin/env python
"""Host-side model of the level path's DRAM rows on the headline circuit (bench.py's generator and seed): how many operand
reads repeat a wire another gate of the same wavefront reads, and how many of them a gate order turns into L2 hits.

A repeat read counts as a hit when the same wire was read within the last K gates of the execution order: K = 2000-5000
stands in for L2 (126 MB = 15 k rows of 8 KB; about 592 resident CTAs of k_level_tma, each 3 items ahead).  DRAM rows per
gate-eval = writes + missed reads, over the algorithmic 3 rows of a two-input gate; every Add/Mul output is counted as
written (the stores F_SINK lets 15 of 16 tiles skip are not modelled).  usage: wavefront_reuse_model.py [log2 gates, 24]
(about 10 minutes at 2^24)."""
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("circuits", os.path.join(ROOT, "zkinterface-ir_b200", "circuits.py"))
c = importlib.util.module_from_spec(spec)
spec.loader.exec_module(c)

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 24
circ = c.random_circuit(1 << lg, 1024, c.BLS12_381_FR, 0x5EED0003)   # bench.py: SEED, --inputs 1024
g = circ.gates
op = g["op"]
a, b, out = g["a"].astype(np.int64), g["b"].astype(np.int64), g["out"].astype(np.int64)
val = np.flatnonzero(np.isin(op, [c.G_ADD, c.G_MUL]))
va, vb, vo, vop = a[val], b[val], out[val], op[val]
# ASAP wavefronts: relax until no level changes
lev = np.zeros(circ.n_wires, np.int32)
for _ in range(300):
    new = 1 + np.maximum(lev[va], lev[vb])
    if (lev[vo] == new).all():
        break
    lev[vo] = new
L = lev[vo].astype(np.int64)
n = val.size
# readers of each operand inside its wavefront
ka, kb = L * (1 << 32) + va, L * (1 << 32) + vb
uk, inv, cnt = np.unique(np.concatenate([ka, kb]), return_inverse=True, return_counts=True)
ma, mb = cnt[inv[:n]], cnt[inv[n:]]
distinct = uk.size


def hits(order, K):
    """order: gate indices in execution order; a gate reads a, then b"""
    pos = np.empty(n, np.int64)
    pos[order] = np.arange(n)
    P, W = np.concatenate([pos, pos]), np.concatenate([va, vb])
    s = np.lexsort((P, W))
    Ws, Ps = W[s], P[s]
    return int(((Ws[1:] == Ws[:-1]) & (Ps[1:] - Ps[:-1] <= K)).sum())


reads = 2 * n
cur = np.lexsort((vo, vop != c.G_ADD, L))                 # value order inside (wavefront, opcode): ZKB_OPERAND_ORDER=0
key = np.where(mb > ma, vb, va)                           # the operand more gates of the wavefront read; a on a tie
prop = np.lexsort((vo, key, L))                           # whole hot range by key
prop2 = np.lexsort((vo, key, vop != c.G_ADD, L))          # by key inside each opcode group: Plan::build's order
print(f"2^{lg}: reads {reads}, in-wavefront duplicates {reads - distinct} ({1 - distinct / reads:.3f} of reads)")
for K in (600, 2000, 5000):
    for name, order in (("current", cur), ("by shared operand", prop), ("by shared operand, opcode split kept", prop2)):
        h = hits(order, K)
        dram = n + reads - h
        print(f"  K={K:5d} {name:40s} read hits {h / reads:.3f}  DRAM rows / algorithmic {dram / (3 * n):.3f}")
