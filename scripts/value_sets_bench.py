"""Value sets from `.sieve` files against the backend's own batch path, on C3 (2^24-gate random Add/Mul/AssertZero circuit
over BLS12-381, 1024 witness inputs, 4096 witnesses, 1 % corrupted: the generator, seeds and corruption bench.py uses).

  A  value sets: Evaluator.add_value_set for each of the 4096 witness files, ingest the relation file, get_batch_violations
     (levelize + upload + one batch on the device)
  B  GpuBackend.evaluate of the same witness array (inputs packed by numpy already) through the same relation, recorded
     by an Evaluator of its own from the relation file and witness file 0 (one statement)

Arms alternate in one process: A then B on even reps, B then A on odd ones, each on a fresh context.  Both must give the same verdicts, and every corrupted witness's violation must name the wire
of the assertion circuits.expected_first_fail predicts.  With two or more devices, A is repeated over all of them.  The card's
name and power limit are printed first.  Usage:  python scripts/value_sets_bench.py [--reps 3]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import zkb_loader  # noqa: E402
from oracle import ir  # noqa: E402
from oracle import sieve_fbs as F  # noqa: E402

SEED = 0x5EED0003             # bench.py


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def witness_file(h, row):
    """one Witness message of the row's values (little-endian bytes, trailing zeros trimmed as a producer writes them)"""
    vals = [bytes(v).rstrip(b"\0") or b"\0" for v in row]
    return F.write_message(ir.Witness(h, vals))


def arm_sets(z, sets_dir, rel_dir, names, sharded=None):
    be = sharded.root if sharded else z.GpuBackend(0)
    e = z.Evaluator(be)
    if sharded:
        e.use_devices(sharded)
    t0 = time.perf_counter()
    for name in names:
        e.add_value_set(z.Source.from_directory(os.path.join(sets_dir, name)))
    t1 = time.perf_counter()
    e.ingest_source(z.Source.from_directory(rel_dir))
    t2 = time.perf_counter()
    res = e.get_batch_violations()
    t3 = time.perf_counter()
    dev_ms = be.timing()["total_ms"]
    return e, res, {"add_sets_s": t1 - t0, "ingest_relation_s": t2 - t1, "levelize_upload_evaluate_s": t3 - t2,
                    "device_ms": dev_ms, "total_s": t3 - t0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2-gates", type=int, default=24)
    ap.add_argument("--witnesses", type=int, default=4096)
    ap.add_argument("--inputs", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    print("card:", card(), flush=True)
    z = zkb_loader.load()
    import importlib
    cm = importlib.import_module("zkir_b200.circuits")
    p = cm.BLS12_381_FR
    n = args.witnesses
    circ = cm.random_circuit(1 << args.log2_gates, args.inputs, p, SEED)
    rng = np.random.default_rng(SEED + 1)
    bad = rng.choice(n, size=max(1, n // 100), replace=False)
    corrupt = {int(j): int(rng.integers(0, max(circ.n_tracked, 1))) for j in bad} if circ.n_tracked else {}
    w = cm.make_witnesses(circ, n, seed=SEED + 7, corrupt=corrupt)
    expected = cm.expected_first_fail(circ, n, corrupt)
    h = ir.Header(p.to_bytes(32, "little"))
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        rel_dir, sets_dir = os.path.join(d, "relation"), os.path.join(d, "sets")
        os.makedirs(rel_dir)
        rel = z.GpuBackend(-1).write_flat_relation(p, circ.gates, circ.const_pool)
        open(os.path.join(rel_dir, "002_relation.sieve"), "wb").write(rel)
        names = [f"w{j:05d}" for j in range(n)]
        wit_bytes = 0
        for j, name in enumerate(names):
            os.makedirs(os.path.join(sets_dir, name))
            b = witness_file(h, w[j])
            wit_bytes += len(b)
            open(os.path.join(sets_dir, name, "001_witness.sieve"), "wb").write(b)
        print(json.dumps({"setup": f"C3 2^{args.log2_gates} gates, BLS12-381, {n} witness files of {args.inputs} values",
                          "relation_bytes": len(rel), "witness_bytes": wit_bytes, "write_s": time.perf_counter() - t0}), flush=True)
        rows = []
        def arm_backend():
            be = z.GpuBackend(0)
            one = z.Evaluator(be)
            t0 = time.perf_counter()
            one.ingest_source(z.Source.from_dirs_and_files([os.path.join(sets_dir, names[0]), rel_dir]))
            assert isinstance(one.get_violations(), list)   # finalizes the program (and runs witness 0)
            t1 = time.perf_counter()
            v = be.evaluate(None, w, n)
            t2 = time.perf_counter()
            return one, v, {"record_levelize_s": t1 - t0, "evaluate_s": t2 - t1, "device_ms": be.timing()["total_ms"]}

        for rep in range(args.reps):
            if rep % 2 == 0:
                e, res, ta = arm_sets(z, sets_dir, rel_dir, names)
                one, v, tb = arm_backend()
            else:
                one, v, tb = arm_backend()
                e, res, ta = arm_sets(z, sets_dir, rel_dir, names)
            be = one.backend
            # same verdicts; corrupted witnesses name the predicted assertion's wire
            n_false = 0
            for j in range(n):
                st, viol = res[j]
                assert st == 0, (j, res[j])
                assert bool(v[j]["ok"]) == (viol == []), (j, viol, v[j])
                want_seq = int(expected[j])
                if want_seq < 0:
                    assert viol == [], (j, viol)
                    continue
                n_false += 1
                assert int(v[j]["first_fail_seq"]) == want_seq, (j, int(v[j]["first_fail_seq"]), want_seq)
                assert viol == [f"Wire_{be.assert_wire(want_seq)} (may be weighted) should be 0, while it is not"], (j, viol)
            assert n_false == len(corrupt), (n_false, len(corrupt))
            row = {"rep": rep, "order": "A,B" if rep % 2 == 0 else "B,A", "value_sets": ta, "backend_evaluate": tb,
                   "verdicts_match": True, "not_true": n_false}
            rows.append(row)
            print(json.dumps(row), flush=True)
            for x in (e, one):
                x.close()
                x.backend.close()
        best = min(rows, key=lambda r: r["value_sets"]["total_s"])
        print(json.dumps({"summary": "best rep by value-set total",
                          "add_sets_s": best["value_sets"]["add_sets_s"],
                          "add_sets_share_of_value_sets_total": best["value_sets"]["add_sets_s"] / best["value_sets"]["total_s"],
                          "value_sets_device_ms": best["value_sets"]["device_ms"],
                          "backend_evaluate_device_ms": best["backend_evaluate"]["device_ms"]}), flush=True)
        import torch
        n_dev = torch.cuda.device_count()
        if n_dev >= 2:
            sb = z.ShardedBackend(list(range(n_dev)))
            e, res, ta = arm_sets(z, sets_dir, rel_dir, names, sharded=sb)
            assert [bool(r[1] == []) for r in res] == [bool(x) for x in v["ok"]]
            print(json.dumps({"devices": n_dev, "value_sets": ta, "verdicts_match": True}), flush=True)
            e.close()
            sb.close()
        else:
            print(json.dumps({"devices": n_dev, "multi_device": "not run (one device)"}), flush=True)


if __name__ == "__main__":
    main()
