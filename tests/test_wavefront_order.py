"""Gate order inside a wavefront (ZKB_OPERAND_ORDER) and skipped sink stores (F_SINK, ZKB_SINK_STORES).

Host: each wavefront's hot range holds the same gates in either order, opcode groups stay contiguous, and inside a group the
gates follow (key operand, value); the F_SINK count is the number of stored values no gate reads; the threaded plan is the
sequential one.  GPU: batches over several tiles, where every tile but the last skips its sink stores, give the oracle's
verdicts for every witness and its wire values — sink wires and assertion sums included — for witnesses of the first, a middle
and the last tile, read in an order that makes earlier tiles resident again."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.util import FIELDS, ROOT, circuits, has_gpu, random_flat_program, zkb

V_WITNESS, V_ADD, V_MUL, V_ADDC, V_MULC, V_AND, V_XOR = 2, 3, 4, 5, 6, 7, 8
F_NOSTORE, F_SINK = 1 << 9, 1 << 12
SWITCHES = {"on": {"ZKB_OPERAND_ORDER": "1", "ZKB_SINK_STORES": "0"},
            "off": {"ZKB_OPERAND_ORDER": "0", "ZKB_SINK_STORES": "1"}}


def _programs():
    c = circuits()
    circ = c.random_circuit(1 << 14, 64, FIELDS["bls381"], seed=3)
    yield FIELDS["bls381"], circ.gates, circ.const_pool
    circ = c.random_circuit(6000, 48, FIELDS["goldilocks"], seed=8, window=500)
    yield FIELDS["goldilocks"], circ.gates, circ.const_pool
    gates, pool, _ = random_flat_program(FIELDS["bn254"], 4000, 5, 9, seed=12, bool_ops=True)   # constants, And / Xor / Not
    yield FIELDS["bn254"], gates, pool


def _plan(z, p, gates, pool, order, keep_all=True):
    os.environ["ZKB_OPERAND_ORDER"] = order
    try:
        b = z.GpuBackend(-1)
        b.set_field(p)
        b.push_gates(gates, pool)
        b.finalize(keep_all_values=keep_all)
    finally:
        del os.environ["ZKB_OPERAND_ORDER"]
    st = b.stats()
    ops, vals = b.plan_ops(values=keep_all) if keep_all else (b.plan_ops(), None)
    levels = [b.level_info(l) for l in range(st["n_levels"])]
    kinds, a, bb = b.program()
    b.close()
    return st, ops, vals, levels, (kinds, a, bb)


def test_hot_range_is_a_permutation_ordered_by_shared_operand():
    z = zkb()
    for p, gates, pool in _programs():
        st0, ops0, vals0, levels, (kinds, a, b) = _plan(z, p, gates, pool, "0")
        st1, ops1, vals1, levels1, _ = _plan(z, p, gates, pool, "1")
        assert levels == levels1 and st0["n_slots"] == st1["n_slots"]
        lo = 0
        moved = 0
        for lv in levels:
            hi = lo + lv["arith"]
            v0, v1 = vals0[lo:hi], vals1[lo:hi]
            assert np.array_equal(np.sort(v0), np.sort(v1))
            op0, op1 = ops0[lo:hi, 3] & 0xFF, ops1[lo:hi, 3] & 0xFF
            assert np.array_equal(op0, op1) and np.all(np.diff(op0.astype(np.int64)) >= 0)   # same contiguous opcode groups
            # rare range untouched
            assert np.array_equal(vals0[hi:lo + lv["gates"]], vals1[hi:lo + lv["gates"]])
            two = np.isin(kinds[v1], [V_ADD, V_MUL])
            reads = np.concatenate([a[v1], b[v1][two]])
            u, cnt = np.unique(reads, return_counts=True)
            readers = lambda w: np.minimum(cnt[np.searchsorted(u, w)], 255)
            key = np.where(two & (readers(np.where(two, b[v1], a[v1])) > readers(a[v1])), b[v1], a[v1])
            for o in np.unique(op1):
                g = op1 == o
                assert np.all(np.diff(v0[g].astype(np.int64)) > 0)              # old order: value order
                order = np.lexsort((v1[g], key[g]))
                assert np.array_equal(order, np.arange(g.sum()))               # new order: (key, value)
            moved += int((v0 != v1).sum())
            lo += lv["gates"]
        assert moved > 0


def test_sink_count_is_the_stored_values_no_gate_reads():
    z = zkb()
    for p, gates, pool in _programs():
        for keep_all in (True, False):
            st, ops, vals, _, (kinds, a, b) = _plan(z, p, gates, pool, "1", keep_all)
            meta = ops[:, 3]
            sink = (meta & F_SINK) != 0
            assert st["n_sink_ops"] == int(sink.sum())
            assert not np.any(sink & ((meta & F_NOSTORE) != 0))
            gate = kinds > V_WITNESS
            two = np.isin(kinds, [V_ADD, V_MUL, V_AND, V_XOR])
            read = np.zeros(len(kinds), dtype=bool)
            read[a[gate]] = True
            read[b[two]] = True
            if keep_all:   # every gate value is stored
                assert st["n_sink_ops"] == int((gate & ~read).sum()) > 0
                assert not read[vals[sink]].any()
            else:
                assert 0 < st["n_sink_ops"] <= int((gate & ~read).sum())


SNIPPET = r'''
import sys, importlib
sys.path.insert(0, %r)
import zkb_loader
z = zkb_loader.load()
c = importlib.import_module("zkir_b200.circuits")
circ = c.random_circuit(1 << 18, 256, c.BLS12_381_FR, 5)
out = []
for keep_all in (False, True):
    b = z.GpuBackend(-1)
    b.set_field(c.BLS12_381_FR)
    b.push_gates(circ.gates, circ.const_pool)
    b.finalize(keep_all_values=keep_all)
    out.append((b.stats()["n_sink_ops"], b.plan_hash()))
print(out)
'''


def _hash(threads, order):
    env = dict(os.environ, ZKB_PLAN_THREADS=str(threads), ZKB_OPERAND_ORDER=order)
    r = subprocess.run([sys.executable, "-c", SNIPPET % ROOT], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr
    return r.stdout.strip().splitlines()[-1]


def test_operand_order_plan_does_not_depend_on_threads():
    on = _hash(1, "1")
    assert on == _hash(6, "1")
    assert on != _hash(6, "0")


# ---- GPU ----------------------------------------------------------------------------------------------------------------
CASES = [  # (field, tile log2, batch, kind): 256-lane tiles of an 8-limb field take k_level_tma, the others k_level_pipe; the
           # flat program's And / Xor / Not gates take k_level<N, true>
    ("bls381", "8", 3 * 256 - 40, "random"),
    ("goldilocks", "5", 100, "random"),
    ("bn254", "2", 11, "flat"),
]


@pytest.mark.gpu
@pytest.mark.skipif(not has_gpu(), reason="needs a GPU")
@pytest.mark.parametrize("switches", list(SWITCHES))
@pytest.mark.parametrize("name,tile_log2,n_batch,kind", CASES)
def test_multi_tile_values_and_verdicts(name, tile_log2, n_batch, kind, switches, monkeypatch):
    from oracle import flat
    c = circuits()
    z = zkb()
    p = FIELDS[name]
    eb = c.elem_bytes(p)
    for k, v in dict(SWITCHES[switches], ZKB_TILE_LOG2=tile_log2, ZKB_COOP="0").items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(n_batch)
    if kind == "random":
        circ = c.random_circuit(1 << 15, 64, p, seed=17, n_tracked=8)
        gates, pool, n_wires, inst = circ.gates, circ.const_pool, circ.n_wires, None
        wit = c.make_witnesses(circ, n_batch, seed=4, corrupt={1: 2, n_batch // 2: 5, n_batch - 1: 0})
    else:
        gates, pool, n_wires = random_flat_program(p, 3000, 5, 9, seed=14, bool_ops=True)
        inst = c.random_field_elements(rng, (n_batch, 5), p)
        wit = c.random_field_elements(rng, (n_batch, 9), p)
    b = z.GpuBackend(0)
    b.set_field(p)
    b.push_gates(gates, pool)
    b.finalize(keep_all_values=False)
    st = b.stats()
    assert st["n_sink_ops"] > 0
    v = b.evaluate(inst, wit, n_batch)
    st = b.stats()
    assert st["n_tiles"] >= 3 and st["tile_witnesses"] == 1 << int(tile_log2)
    ref = flat.eval_batch(gates, pool, p.to_bytes(eb, "little"), inst, wit, n_batch, n_threads=4)
    for j in range(n_batch):
        ok_ref = int(ref[j]["status"]) == flat.EV_TRUE
        assert bool(v[j]["ok"]) == ok_ref, (j, v[j], ref[j])
        if not ok_ref:
            assert int(v[j]["first_fail_seq"]) == int(ref[j]["fail_assert_seq"]), (j, v[j], ref[j])
    if kind == "flat":   # its last assertion almost surely fails: the reference defines no wire values to compare
        b.close()
        return
    tw = st["tile_witnesses"]
    good = [j for j in range(n_batch) if int(ref[j]["status"]) == flat.EV_TRUE]
    first = good[0]
    middle = next(j for j in good if j >= tw * (st["n_tiles"] // 2))
    last = good[-1]
    assert first < tw and last >= tw * (st["n_tiles"] - 1)
    for j in (last, first, middle, last, first):   # the last tile is resident after the run; the others are re-run
        _, dump = flat.eval_dump(gates, pool, p.to_bytes(eb, "little"), None if inst is None else inst[j], wit[j], n_wires,
                                 stride=eb)
        live = [i for i in range(n_wires) if not (dump[i] == 0xFF).all()]
        got = b.read_values(j, [b.scope_lookup(i) for i in live], eb)
        assert got == [int.from_bytes(dump[i].tobytes(), "little") for i in live], j
    b.close()
