"""Full-size (or near full-size) runs of BASELINE.json's configs, checked through properties that do not need the oracle
to replay the whole circuit: verdicts against witnesses corrupted at known assertions (C2, C3), first violated row of a
perturbed R1CS assignment (C4), probe outputs of the unrolled nested-For relation (C5).  The timed variants of the
same checks are tests/bench_configs.py and bench.py."""
import importlib
import os
import sys

import numpy as np
import pytest

from tests.util import ROOT, circuits, zkb

pytestmark = pytest.mark.gpu


def _bc():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    return importlib.import_module("bench_configs")


def test_c2_full_size_goldilocks_single_witness():
    out = _bc().c2(20, 0)                       # asserts the corrupted witness fails at the constructed assertion
    assert out["levels"] > 10 and out["gates_per_s"] > 0


def test_c3_2p22_gates_bls_batch_with_corrupted_witnesses():
    c = circuits()
    z = zkb()
    p = c.BLS12_381_FR
    circ = c.random_circuit(1 << 22, 1024, p, 0x5EED0003)
    n = 96
    rng = np.random.default_rng(3)
    corrupt = {int(j): int(rng.integers(0, circ.n_tracked)) for j in rng.choice(n, size=9, replace=False)}
    w = c.make_witnesses(circ, n, seed=5, corrupt=corrupt)
    b = z.GpuBackend(0)
    b.set_field(p)
    b.push_gates(circ.gates, circ.const_pool)
    b.finalize()
    v = b.evaluate(None, w, n)
    exp = c.expected_first_fail(circ, n, corrupt)
    got = [(-1 if x["ok"] else int(x["first_fail_seq"])) for x in v]
    assert got == list(exp)
    # idempotence: the resident inputs give the same verdicts again; verdicts-only planning agrees
    assert [(-1 if x["ok"] else int(x["first_fail_seq"])) for x in b.run()] == got
    b2 = z.GpuBackend(0)
    b2.set_field(p)
    b2.push_gates(circ.gates, circ.const_pool)
    b2.finalize(verdicts_only=True)
    assert [(-1 if x["ok"] else int(x["first_fail_seq"])) for x in b2.evaluate(None, w, n)] == got
    assert b2.stats()["n_slots"] < b.stats()["n_slots"]


def test_c3_headline_shape_wire_values_2p24_gates_two_tiles():
    """BASELINE.json's C3 relation itself (2^24 gates, BLS12-381 Fr, ~15.3 M wire-store slots) with 512 witnesses = two
    tiles of 256: more than 10^4 wire values spread over every level, for lane 0, both sides of the tile boundary and the
    last lane, bit-exact against the oracle's evaluation of the whole relation; verdicts of all 512 witnesses against the
    generator's expectation, and a corrupted witness's first failing assertion against the oracle."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import flat
    c = circuits()
    z = zkb()
    p = c.BLS12_381_FR
    circ = c.random_circuit(1 << 24, 1024, p, 0x5EED0003)
    n = 512
    corrupt = {7: 3, 255 - 8: 11, 256 + 5: 0, 500: 31}
    w = c.make_witnesses(circ, n, seed=17, corrupt=corrupt)
    b = z.GpuBackend(0)
    b.set_field(p)
    b.push_gates(circ.gates, circ.const_pool)
    b.finalize()
    v = b.evaluate(None, w, n)
    st = b.stats()
    assert st["tile_witnesses"] == 256 and st["n_tiles"] == 2, st
    got = [(-1 if x["ok"] else int(x["first_fail_seq"])) for x in v]
    assert got == list(c.expected_first_fail(circ, n, corrupt))
    picks = [0, 255, 256, 511, 7]           # the last one is corrupted: the oracle stops at its first failing assertion
    mod_le = p.to_bytes(32, "little")
    nw = circ.n_wires
    with ThreadPoolExecutor(len(picks)) as ex:
        dumps = list(ex.map(lambda j: flat.eval_dump(circ.gates, circ.const_pool, mod_le, None, w[j], nw), picks))
    res7 = dumps[-1][0]
    assert int(res7["status"]) == flat.EV_ASSERT_FAILED and int(res7["fail_assert_seq"]) == got[7]
    assert b.assert_wire(got[7]) == int(res7["fail_wire"])
    wires = np.unique(np.concatenate([np.linspace(0, nw - 1, 12000).astype(np.int64), np.arange(nw - 1000, nw), np.arange(64)]))
    handles = [b.scope_lookup(int(i)) for i in wires]
    assert len(wires) > 10000
    for j, (res, dump) in zip(picks[:4], dumps[:4]):
        assert int(res["status"]) == flat.EV_TRUE
        vals = b.read_values(j, handles, 32)
        want = [int.from_bytes(dump[i].tobytes(), "little") for i in wires]
        assert vals == want, (j, [int(wires[q]) for q in range(len(wires)) if vals[q] != want[q]][:5])
    b.close()


def test_c4_2p20_rows_bn254_first_violated_row():
    out = _bc().c4(20, 18, 1)                   # asserts ok for the satisfying z and the first violated row for a perturbed one
    assert out["constraints_per_s"] > 0
    out = _bc().c4(16, 14, 64)
    assert out["constraints_per_s"] > 0


def test_c5_2p22_leaf_gates_nested_for_probe_outputs():
    out = _bc().c5(10, 9, 64)                   # checks verdicts and probe wires against an independent numpy evaluation
    assert out["levels"] > 0


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """bench.py --dump-outputs: the last timed step's verdicts and sampled wire values as float64 .npy files, consistent
    with the JSON line, and identical across two runs with the same arguments (the inputs are seeded)"""
    import json
    import subprocess
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", str(k),
                            "--log2-gates", "14", "--witnesses", "300", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        line = json.loads(r.stdout.strip())
        assert line["steps"] == 2 and line["warmup"] == k
        files = {f.name: np.load(f) for f in d.iterdir()}
        assert sorted(files) == ["first_fail_seq.npy", "verdict_ok.npy", "wire_values.npy"]
        assert all(a.dtype == np.float64 for a in files.values()) and sum(a.nbytes for a in files.values()) <= 64 << 20
        ok, ff = files["verdict_ok.npy"], files["first_fail_seq.npy"]
        assert ok.shape == ff.shape == (300,)
        assert int(ok.sum()) == line["verdicts"]["true"] and int((ok == 0).sum()) == line["verdicts"]["false"] > 0
        assert ((ok == 1) == (ff == -1)).all()
        wv = files["wire_values.npy"]
        assert wv.shape[0] == 16 and wv.shape[2] == 8 and (wv >= 0).all() and (wv < 2 ** 32).all() and wv.any()
        dumps.append(files)
    for name in dumps[0]:
        assert np.array_equal(dumps[0][name], dumps[1][name]), name
