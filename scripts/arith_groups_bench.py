"""C6: loop-structured recording over a prime field, grouped (k_arith_groups) against unrolled (ZKB_NO_CALL_GROUPS=1).

Statement: witnesses 0 .. 2^13-1; an anonymous outer `For i` over 2^L1 whose body runs an inner `For j` over 2^L2 calls of
`round3`, a function of 4 inputs (x0, x1, x2, w) and 3 outputs: 3 rounds of round constants, an x^5 S-box on 3 elements and a
3x3 MulConstant mix (27 gates each), plus one check AssertZero((x0+1)^2 - x0^2 - 2 x0 - 1 - w) (10 gates + the assertion).
Call (i, j) reads x_k = witness[2048 k + i + j] and w = witness[6144 + i + j]: w is 0 on good witnesses, and a witness whose
w at 6144 + m is corrupted first fails in call (i, j) = (max(0, m - 2^L2 + 1), m - i), sequence i * 2^L2 + j.

Both arms are recorded, planned and run in one process, alternating; per arm the script prints one JSON line: host
preparation (ingest + finalize + one single-witness evaluation), GateOp bytes, n_values, tile width, gate-evals/s over the timed runs, and the parity of
verdicts, first failures and a seeded sample of call outputs on several witnesses between the arms.  The card's name and
power limit are printed first.  Usage:  python scripts/arith_groups_bench.py [--fields bls12_381,p127,goldilocks]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ir  # noqa: E402
from oracle import sieve_fbs as F  # noqa: E402

FIELDS = {"bls12_381": 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001,
          "p127": 2**127 - 1, "goldilocks": 2**64 - 2**32 + 1}
N_WIT = 1 << 13
I, C = (lambda n: ("Name", n)), (lambda v: ("Const", v))
add = lambda l, r: ("Add", l, r)


def round3(p, nb):
    le = lambda v: (v % p).to_bytes(nb, "little")
    rng = np.random.default_rng(6)
    rc = lambda: int.from_bytes(rng.bytes(nb + 8), "little") % p
    g = []
    nxt = [7]

    def new():
        nxt[0] += 1
        return nxt[0] - 1
    x0, x1, x2, w = 3, 4, 5, 6
    # check: (x0+1)^2 - x0^2 - 2 x0 - 1 - w == 0
    t = new(); g.append(("AddConstant", t, x0, le(1)))
    t2 = new(); g.append(("Mul", t2, t, t))
    s = new(); g.append(("Mul", s, x0, x0))
    u = new(); g.append(("MulConstant", u, s, le(-1)))
    v = new(); g.append(("Add", v, t2, u))
    d = new(); g.append(("MulConstant", d, x0, le(-2)))
    v2 = new(); g.append(("Add", v2, v, d))
    v3 = new(); g.append(("AddConstant", v3, v2, le(-1)))
    wn = new(); g.append(("MulConstant", wn, w, le(-1)))
    z = new(); g.append(("Add", z, v3, wn))
    g.append(("AssertZero", z))
    st = [x0, x1, x2]
    for r in range(3):
        a = []
        for k in range(3):
            y = new(); g.append(("AddConstant", y, st[k], le(rc())))
            y2 = new(); g.append(("Mul", y2, y, y))
            y4 = new(); g.append(("Mul", y4, y2, y2))
            y5 = new(); g.append(("Mul", y5, y4, y))
            a.append(y5)
        out = []
        for k in range(3):
            m = [new() for _ in range(3)]
            for q in range(3):
                g.append(("MulConstant", m[q], a[q], le(rc())))
            s1 = new(); g.append(("Add", s1, m[0], m[1]))
            dst = k if r == 2 else new()
            g.append(("Add", dst, s1, m[2]))
            out.append(dst)
        st = out
    return ir.Function("round3", 3, 4, 0, 0, g), sum(1 for x in g)


def relation(p, l1, l2):
    nb = (p.bit_length() + 7) // 8
    h = ir.Header(p.to_bytes(nb, "little"))
    fn, body = round3(p, nb)
    n_in, n_out = 1 << l2, 1 << l1
    gates = [("For", "k", 0, N_WIT - 1, [ir.WireRange(0, N_WIT - 1)],
              ("IterExprAnonCall", [("Single", I("k"))], [], 0, 1, [("Witness", 0)]))]
    block = 3 * n_in   # outer body: outputs local 0 .. block-1, inputs (all witnesses) local block .. block + N_WIT - 1
    ins = [("Single", add(add(C(block + off), I("i")), I("j"))) for off in (0, 2048, 4096, 6144)]
    inner = ("For", "j", 0, n_in - 1, [ir.WireRange(0, block - 1)],
             ("IterExprCall", "round3", [("Range", ("Mul", I("j"), C(3)), add(("Mul", I("j"), C(3)), C(2)))], ins))
    base = N_WIT
    gates.append(("For", "i", 0, n_out - 1, [ir.WireRange(base, base + n_out * block - 1)],
                  ("IterExprAnonCall",
                   [("Range", add(C(base), ("Mul", I("i"), C(block))), add(C(base + block - 1), ("Mul", I("i"), C(block))))],
                   [("Range", C(0), C(N_WIT - 1))], 0, 0, [inner])))
    rel = ir.Relation(h, ir.ARITH, ir.FOR | ir.FUNCTION, [fn], gates)
    return rel, nb, body, base, n_out * block


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def run_arm(z, msgs_buf, grouped, W, n_batch, steps, sample_wires, probe):
    if grouped:
        os.environ.pop("ZKB_NO_CALL_GROUPS", None)
    else:
        os.environ["ZKB_NO_CALL_GROUPS"] = "1"
    t0 = time.perf_counter()
    b = z.GpuBackend(0)
    e = z.Evaluator(b)
    e.ingest_source(z.Source.from_buffers([msgs_buf]))
    assert e.get_violations() == []   # the Evaluator's own finalize (its live wires stay readable) + one all-zero witness
    prep = time.perf_counter() - t0
    os.environ.pop("ZKB_NO_CALL_GROUPS", None)
    st = b.stats()
    b.upload_inputs(None, W, n_batch)
    v = b.run()   # warm-up
    times = []
    for _ in range(steps):
        t = time.perf_counter()
        v = b.run()
        times.append(time.perf_counter() - t)
    st = b.stats()
    hs = [e.value_handle(x) for x in sample_wires]
    vals = [b.read_values(j, hs, 32) for j in probe]
    res = {"arm": "grouped" if grouped else "unrolled", "host_prep_s": round(prep, 3),
           "gateop_bytes": int(st["n_device_ops"]) * 16, "n_values": int(st["n_values"]),
           "n_call_groups": int(st["n_call_groups"]), "tile_witnesses": int(st["tile_witnesses"]),
           "step_s_median": float(np.median(times)), "step_s_min": float(min(times)),
           "gate_evals_per_s": float(st["ir_gates"]) * n_batch / float(np.median(times))}
    out = (v["ok"].copy(), v["first_fail_seq"].copy(), vals)
    b.close()
    return res, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fields", default="bls12_381,p127,goldilocks")
    ap.add_argument("--witnesses", type=int, default=4096)
    ap.add_argument("--log2-outer", type=int, default=10)
    ap.add_argument("--log2-inner", type=int, default=10)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2, help="grouped / unrolled alternations per field")
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    from tests.util import zkb
    z = zkb()
    print(json.dumps({"card": card()}), flush=True)
    for fname in a.fields.split(","):
        p = FIELDS[fname]
        rel, nb, body, out_base, n_outs = relation(p, a.log2_outer, a.log2_inner)
        n_batch = a.witnesses
        rng = np.random.default_rng(1)
        top = max(1, (p.bit_length() - 2) - 8 * (nb - 1))   # values below 2^(bits-2) < p
        W = rng.integers(0, 256, size=(n_batch, N_WIT, nb), dtype=np.uint8)
        W[:, :, nb - 1] &= np.uint8((1 << top) - 1)
        W[:, 6144:, :] = 0
        bad = rng.choice(n_batch, max(1, n_batch // 100), replace=False)
        n_calls_in = 1 << a.log2_inner
        limit = (1 << a.log2_outer) - 1 + n_calls_in - 1
        expect = {}
        for j in bad:
            m = int(rng.integers(0, min(limit, N_WIT - 6144 - 1) + 1))
            W[j, 6144 + m, 0] = 1
            i = max(0, m - n_calls_in + 1)
            expect[int(j)] = i * n_calls_in + (m - i)
        buf = F.write_messages([ir.Witness(rel.header, [bytes(nb)] * N_WIT), rel])
        sample = [int(out_base + x) for x in rng.choice(n_outs, 256, replace=False)]
        good = [int(j) for j in range(n_batch) if j not in expect]
        probe = [good[0], good[len(good) // 2], good[-1], int(bad[0])]
        ref = None
        for rnd in range(a.rounds):
            for grouped in (True, False):
                res, out = run_arm(z, buf, grouped, W, n_batch, a.steps, sample, probe)
                res.update({"field": fname, "limbs": {32: 8, 16: 4, 8: 2}[nb], "round": rnd, "witnesses": n_batch,
                            "calls": (1 << a.log2_outer) << a.log2_inner, "body_gates": body})
                ff = out[1]
                res["known_first_failures_ok"] = all(int(ff[j]) == s for j, s in expect.items()) and \
                    all(bool(out[0][j]) for j in good)
                if ref is None:
                    ref = out
                else:
                    res["verdict_parity"] = bool((out[0] == ref[0]).all() and (out[1] == ref[1]).all())
                    res["sample_parity"] = out[2] == ref[2]
                print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
