"""C7: carried loops over a prime field, grouped (k_arith_chain) against unrolled (ZKB_NO_CALL_GROUPS=1).

Statement: witnesses w_0 .. w_{2n+2}; a Horner chain acc_i = acc_{i-1} * x + w_i over a named function (seed w_{2n+1}, x =
w_{2n}) and a grand-product check g_i = g_{i-1} * w_i, AssertZero(g_i - w_{n+i}) over an anonymous body (seed w_{2n+2}),
n calls each, and one gate after the loops that adds their last outputs.  Unrolled, each chain is 2n dependent wavefronts
one gate wide; grouped, one thread per witness walks the calls.  Witness j % 97 == 5 has b_i off by one at step (j * 7919) % n,
so its first failure is that step's assertion.

Both arms are recorded, planned and run in one process, alternating; per arm the script prints one JSON line: host
preparation (ingest + finalize + one evaluation of the recording's witness), step time, gate-evals/s, and the parity of
verdicts, first failures and sampled chain outputs against the first arm run and against the values computed here.  The
arms alternate --rounds times per point.  The unrolled arm stops after the first size whose step took longer than
--unrolled-limit seconds; points whose witness array exceeds --max-input-gb are listed as skipped, with the size.  The card's name and power
limit are printed first.  Usage:  python scripts/chain_groups_bench.py [--fields ...] [--log2-calls 12,16,20] [--witnesses 1,4096]"""
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
I, C = (lambda n: ("Name", n)), (lambda v: ("Const", v))
add = lambda l, r: ("Add", l, r)
mul = lambda l, r: ("Mul", l, r)


def relation(p, n):
    nb = (p.bit_length() + 7) // 8
    h = ir.Header(p.to_bytes(nb, "little"))
    n_wit = 2 * n + 3
    horner = ir.Function("horner", 1, 3, 0, 0, [("Mul", 4, 1, 2), ("Add", 0, 4, 3)])
    prod = [("Mul", 0, 1, 2), ("MulConstant", 4, 3, (p - 1).to_bytes(nb, "little")), ("Add", 5, 0, 4), ("AssertZero", 5)]
    gates = [("For", "k", 0, n_wit - 1, [ir.WireRange(0, n_wit - 1)],
             ("IterExprAnonCall", [("Single", I("k"))], [], 0, 1, [("Witness", 0)]))]
    hb = n_wit + 1        # horner outputs hb + i; its seed (wire hb - 1) is a copy of w_{2n+1}
    gates.append(("Copy", hb - 1, 2 * n + 1))
    gates.append(("For", "i", 0, n - 1, [ir.WireRange(hb, hb + n - 1)],
                  ("IterExprCall", "horner", [("Single", add(C(hb), I("i")))],
                   [("Single", add(C(hb - 1), I("i"))), ("Single", C(2 * n)), ("Single", I("i"))])))
    gb = hb + n + 1
    gates.append(("Copy", gb - 1, 2 * n + 2))
    gates.append(("For", "i", 0, n - 1, [ir.WireRange(gb, gb + n - 1)],
                  ("IterExprAnonCall", [("Single", add(C(gb), I("i")))],
                   [("Single", add(C(gb - 1), I("i"))), ("Single", I("i")), ("Single", add(C(n), I("i")))], 0, 0, prod)))
    gates.append(("Add", gb + n, hb + n - 1, gb + n - 1))
    rel = ir.Relation(h, ir.ARITH, ir.FOR | ir.FUNCTION, [horner], gates)
    return rel, nb, n_wit, hb, gb


def witness_rows(p, n, nb, n_batch, rng):
    """values < 2^62, x = w_{2n} different per witness; returns the uint8 array, the sampled horner / product values of
    witness 0 and the expected first failures"""
    v = [int(x) for x in rng.integers(1, 1 << 62, size=(2 * n + 3,), dtype=np.int64)]
    prods, g = [], v[2 * n + 2]
    for i in range(n):
        g = g * v[i] % p
        prods.append(g)
    v[n:2 * n] = prods
    row = np.frombuffer(b"".join(x.to_bytes(nb, "little") for x in v), dtype=np.uint8).reshape(-1, nb)
    W = np.repeat(row[None], n_batch, axis=0)
    expect = {}
    for j in range(n_batch):
        W[j, 2 * n] = np.frombuffer((v[2 * n] + j).to_bytes(nb, "little"), dtype=np.uint8)
        if j % 97 == 5:
            s = (j * 7919) % n
            W[j, n + s] = np.frombuffer(((prods[s] + 1) % p).to_bytes(nb, "little"), dtype=np.uint8)
            expect[j] = s
    hs, acc = {}, v[2 * n + 1]
    for i in range(n):
        acc = (acc * v[2 * n] + v[i]) % p
        if i in SAMPLE_AT(n):
            hs[i] = acc
    return W, hs, {i: prods[i] for i in SAMPLE_AT(n)}, expect


def SAMPLE_AT(n):
    return {0, 1, n // 3, n // 2, n - 2, n - 1}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def run_arm(z, buf, grouped, W, n_batch, steps, wires, probe):
    if grouped:
        os.environ.pop("ZKB_NO_CALL_GROUPS", None)
    else:
        os.environ["ZKB_NO_CALL_GROUPS"] = "1"
    t0 = time.perf_counter()
    b = z.GpuBackend(0)
    e = z.Evaluator(b)
    e.ingest_source(z.Source.from_buffers([buf]))
    e.get_violations()   # the Evaluator's own finalize and one evaluation of the recorded witness
    prep = time.perf_counter() - t0
    os.environ.pop("ZKB_NO_CALL_GROUPS", None)
    b.upload_inputs(None, W, n_batch)
    v = b.run()   # warm-up
    times = []
    for _ in range(steps):
        t = time.perf_counter()
        v = b.run()
        times.append(time.perf_counter() - t)
    st = b.stats()
    hs = [e.value_handle(x) for x in wires]
    vals = [b.read_values(j, hs, 32) for j in probe]
    res = {"arm": "grouped" if grouped else "unrolled", "host_prep_s": round(prep, 3), "n_values": int(st["n_values"]),
           "n_call_groups": int(st["n_call_groups"]), "n_carried_groups": int(st["n_carried_groups"]),
           "n_levels": int(st["n_levels"]), "tile_witnesses": int(st["tile_witnesses"]),
           "step_s_median": float(np.median(times)), "step_s_min": float(min(times)),
           "gate_evals_per_s": float(st["ir_gates"]) * n_batch / float(np.median(times))}
    out = (v["ok"].copy(), v["first_fail_seq"].copy(), vals)
    b.close()
    return res, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fields", default="bls12_381,p127,goldilocks")
    ap.add_argument("--log2-calls", default="12,16,20")
    ap.add_argument("--witnesses", default="1,4096")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--unrolled-limit", type=float, default=60.0, help="seconds per step after which larger unrolled sizes are skipped")
    ap.add_argument("--rounds", type=int, default=2, help="grouped / unrolled alternations per point")
    ap.add_argument("--max-input-gb", type=float, default=24.0,
                    help="skip points whose witness array is larger (each skipped point is listed with its size)")
    a = ap.parse_args()
    from tests.util import zkb
    z = zkb()
    print(json.dumps({"card": card()}), flush=True)
    for fname in a.fields.split(","):
        p = FIELDS[fname]
        for n_batch in [int(x) for x in a.witnesses.split(",")]:
            unrolled_ok = True
            for l2 in [int(x) for x in a.log2_calls.split(",")]:
                n = 1 << l2
                rel, nb, n_wit, hb, gb = relation(p, n)
                gb_in = n_batch * n_wit * nb / 1e9
                point = {"field": fname, "limbs": {32: 8, 16: 4, 8: 2}[nb], "witnesses": n_batch, "calls_per_chain": n}
                if gb_in > a.max_input_gb:
                    print(json.dumps(dict(point, skipped=f"witness array of {gb_in:.1f} GB")), flush=True)
                    continue
                rng = np.random.default_rng(l2)
                W, hs_ref, gs_ref, expect = witness_rows(p, n, nb, n_batch, rng)
                buf = F.write_messages([ir.Witness(rel.header, [bytes(W[0, k]) for k in range(n_wit)]), rel])
                at = sorted(SAMPLE_AT(n))
                wires = [hb + i for i in at] + [gb + i for i in at] + [gb + n]
                good = [j for j in range(n_batch) if j not in expect]
                probe = sorted(set([0, good[len(good) // 2], n_batch - 1]))
                ref = None
                for rnd, grouped in [(r, g) for r in range(a.rounds) for g in (True, False)]:
                    if not grouped and not unrolled_ok:
                        print(json.dumps(dict(point, arm="unrolled", skipped="a smaller size ran past --unrolled-limit")), flush=True)
                        continue
                    res, out = run_arm(z, buf, grouped, W, n_batch, a.steps, wires, probe)
                    res.update(point, round=rnd)
                    ff = out[1]
                    res["known_first_failures_ok"] = all(int(ff[j]) == s for j, s in expect.items()) and all(bool(out[0][j]) for j in good)
                    w0 = out[2][0]
                    res["values_ok"] = [w0[k] for k in range(len(at))] == [hs_ref[i] for i in at] and \
                        [w0[len(at) + k] for k in range(len(at))] == [gs_ref[i] for i in at]
                    if ref is None:
                        ref = out
                    else:
                        res["verdict_parity"] = bool((out[0] == ref[0]).all() and (out[1] == ref[1]).all())
                        res["sample_parity"] = out[2] == ref[2]
                    print(json.dumps(res), flush=True)
                    if not grouped and res["step_s_median"] > a.unrolled_limit:
                        unrolled_ok = False


if __name__ == "__main__":
    main()
