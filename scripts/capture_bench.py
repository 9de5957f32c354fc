"""Cost of a capture list on C3 (2^24-gate random Add/Mul/AssertZero circuit over BLS12-381, 4096 witnesses, the generator
and seed bench.py uses), one GPU, inputs resident, arms alternated in one process:

  A  verdicts only (no list)
  B  the 4096 wires of bench.py --dump-outputs' sample, captured for all 4096 witnesses
  C  every live output wire (a wire no gate reads); when their bytes do not fit in device memory the run is refused with
     ZKB_E_CUDA (reported), and C runs the largest prefix of them that fits --c-max-gb
  D  the per-witness zkb_read_values loop over B's wires, for all 4096 witnesses

B is checked against D bit for bit.  Step times are the library's device events around a run (zkb_get_timing total_ms).
The card's name and power limit are printed first.  Usage:  python scripts/capture_bench.py [--steps 3] [--reps 3]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import zkb_loader  # noqa: E402

SEED = 0x5EED0003             # bench.py
DUMP_WIRES = 4096             # bench.py --dump-outputs
G_ADD, G_MUL, G_ADD_CONSTANT, G_MUL_CONSTANT, G_ASSERT_ZERO, G_COPY = 4, 5, 6, 7, 2, 3


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2-gates", type=int, default=24)
    ap.add_argument("--witnesses", type=int, default=4096)
    ap.add_argument("--inputs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--c-max-gb", type=float, default=16.0)
    args = ap.parse_args()
    print("card:", card(), flush=True)
    z = zkb_loader.load()
    import importlib
    cm = importlib.import_module("zkir_b200.circuits")
    p = cm.BLS12_381_FR
    eb = cm.elem_bytes(p)
    t0 = time.perf_counter()
    circ = cm.random_circuit(1 << args.log2_gates, args.inputs, p, SEED)
    be = z.GpuBackend(0)
    be.set_field(p)
    be.push_gates(circ.gates, circ.const_pool)
    be.finalize()
    n = args.witnesses
    w = cm.make_witnesses(circ, n, seed=SEED + 7, corrupt={})
    be.upload_inputs(None, w, n)
    print(f"prepared in {time.perf_counter() - t0:.1f} s; {be.stats()['n_tiles']} tiles of {be.stats()['tile_witnesses']}", flush=True)

    rng = np.random.default_rng(SEED + 11)
    wires_b = np.sort(rng.choice(circ.n_wires, size=min(DUMP_WIRES, circ.n_wires), replace=False))
    hb = [be.scope_lookup(int(i)) for i in wires_b]
    g = circ.gates
    reads_a = np.isin(g["op"], [G_ADD, G_MUL, G_ADD_CONSTANT, G_MUL_CONSTANT, G_ASSERT_ZERO, G_COPY])
    read = np.zeros(circ.n_wires, dtype=bool)
    read[g["a"][reads_a]] = True
    read[g["b"][np.isin(g["op"], [G_ADD, G_MUL])]] = True
    outputs = np.flatnonzero(~read)
    per_wire = n * eb
    fit = int(args.c_max_gb * (1 << 30) // per_wire)
    print(f"live output wires: {len(outputs)} ({len(outputs) * per_wire / 1e9:.1f} GB for {n} witnesses)", flush=True)
    hc_all = [be.scope_lookup(int(i)) for i in outputs]
    c_refused = None
    if len(hc_all) > fit:
        be.capture(hc_all)
        try:
            be.run()
        except z.ZkbError as e:
            c_refused = f"code {e.code}: {e}"
            print("C (every output) refused:", c_refused, flush=True)
    hc = hc_all[:fit]

    arms = {"A": [], "B": hb, "C": hc}
    res = {k: [] for k in arms}
    verdicts = {}
    for rep in range(args.reps):
        for name, hs in arms.items():
            be.capture(hs)
            verdicts[name] = be.run()            # warm-up (and the first touch of the capture buffer)
            ms = []
            for _ in range(args.steps):
                be.run()
                ms.append(be.timing()["total_ms"])
            res[name] += ms
            print(f"rep {rep} {name}: {len(hs)} values, step ms {['%.2f' % x for x in ms]}", flush=True)
    assert all(np.array_equal(verdicts["A"], v) for v in verdicts.values()), "verdicts differ between arms"

    be.capture(hb)
    be.run()
    t0 = time.perf_counter()
    cap = be.read_captured(0, n, eb)
    t_read = time.perf_counter() - t0
    t0 = time.perf_counter()
    d = np.zeros_like(cap)
    for j in range(n):
        d[j] = [np.frombuffer(x.to_bytes(eb, "little"), np.uint8) for x in be.read_values(j, hb, eb)]
    t_d = time.perf_counter() - t0
    same = bool(np.array_equal(cap, d))
    a = float(np.median(res["A"]))
    out = {
        "card": card(), "workload": f"C3: 2^{args.log2_gates} gates, BLS12-381, {n} witnesses",
        "step_ms_median": {k: float(np.median(v)) for k, v in res.items()},
        "step_ms_all": res,
        "captured_bytes": {"B": len(hb) * per_wire, "C": len(hc) * per_wire},
        "ratio_to_A": {k: float(np.median(v)) / a for k, v in res.items()},
        "C_every_output": {"values": len(hc_all), "bytes": len(hc_all) * per_wire, "refused": c_refused},
        "read_captured_B_s": t_read, "D_read_values_loop_s": t_d, "B_equals_D": same,
    }
    print(json.dumps(out), flush=True)
    assert same, "captured values differ from the read_values loop"


if __name__ == "__main__":
    main()
