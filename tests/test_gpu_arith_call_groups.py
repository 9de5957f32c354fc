"""Call groups over prime fields on the device (kernels.cu: k_arith_groups): verdicts, first failing assertions, violation
texts and every readable value against oracle/evaluator.py, and bit-for-bit parity with the gate-by-gate recording
(ZKB_NO_CALL_GROUPS=1) over batches, tiles, sharded contexts and the `evaluate` command line."""
import os
import subprocess

import numpy as np
import pytest

from oracle import evaluator as ev
from oracle import ir
from oracle import sieve_fbs as F
from tests.test_arith_call_groups_host import (BLS12_381_FR, FIELDS, GOLDILOCKS, MIN_CALLS, P101, P127, ArithRel, build,
                                               record)
from tests.util import zkb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "zkinterface-ir_b200", "zkb")


def witness_array(r, ws):
    return np.array([[list(r.le(x % (1 << (8 * r.nb)))) for x in w] for w in ws], dtype=np.uint8)


def check_against_oracle(r, w):
    msgs = r.messages(w)
    expected = ev.evaluate(msgs)
    b, e = record(0, msgs)
    assert b.stats()["n_call_groups"] >= 1
    b.finalize(True)
    assert e.get_violations() == expected
    assert b.stats()["group_jit_state"] == -1
    if expected == []:
        o = ev.Evaluator.from_messages(msgs, ev.PlaintextBackend())
        for wid, val in o.values.items():
            assert e.get(wid) == val, wid
    return b, e


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(FIELDS))
@pytest.mark.parametrize("seed", [0, 1])
def test_gpu_values_and_verdicts(field, seed):
    r = build(FIELDS[field], seed, n_asserts=1)
    check_against_oracle(r, r.witness())


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(FIELDS))
def test_gpu_raw_witness_values_feed_groups(field):
    """witness values >= p (the reference keeps them unreduced) as call inputs: Add / Mul inside the call reduce them"""
    r = build(FIELDS[field], 50, raw=True, n_asserts=1)
    w = r.witness()
    assert any(x >= r.p for x in w)
    check_against_oracle(r, w)


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(FIELDS))
def test_gpu_failing_assertion_on_a_group_output(field):
    r = build(FIELDS[field], 60, failing=True)
    for trial in range(2):
        msgs = r.messages(r.witness())
        b, e = record(0, msgs)
        assert e.get_violations() == ev.evaluate(msgs)


def operand_forms(p):
    """groups reading groups (depth 1 and 2), stride-0 inputs and slot-table inputs"""
    r = ArithRel(p, 9)
    f = r.function("f", 2, 3, "plain", 1)
    g = r.function("g", 1, 2, "plain", 2)
    r.witnesses()
    tb = r.table_witnesses(MIN_CALLS + 2)
    b1, s1 = r.loop(f, n_calls=MIN_CALLS, in_specs=[(0, 1), (3, 0), (tb, 2)])
    b2, _ = r.loop(g, n_calls=MIN_CALLS, in_specs=[(b1, s1), (7, 0)])
    r.loop(g, n_calls=MIN_CALLS + 1, in_specs=[(b2, 0), (1, 1)])
    r.tail()
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(FIELDS))
def test_gpu_operand_forms(field):
    r = operand_forms(FIELDS[field])
    b, e = check_against_oracle(r, r.witness())
    st = b.stats()
    assert st["n_call_groups"] == 3 and st["n_group_launches"] >= 2 and st["n_group_table_slots"] > 0


def order_relation(p):
    """witness block of zeros; f's two assertions test its inputs (through a computed copy): call c's k-th fails when the
    witness read as its input k is non-zero.  One assertion before the loop (witness 1200), one after (witness 1201)."""
    r = ArithRel(p, 3, n_wit=1210)
    one = r.le(1)
    # wires: output 0, inputs 1, 2; k = 0 tests input 0, k = 1 input 1
    body = [("Mul", 3, 1, 2), ("Add", 0, 3, 1), ("MulConstant", 4, 1, one), ("AssertZero", 4),
            ("MulConstant", 5, 2, one), ("AssertZero", 5)]
    r.funcs.append(ir.Function("chk", 1, 2, 0, 0, body))
    r.witnesses()
    s = r.next
    r.gates += [("MulConstant", s, 1200, one), ("AssertZero", s)]
    r.next += 1
    r.loop(("chk", 1, 2, "plain"), n_calls=MIN_CALLS, in_specs=[(0, 1), (100, 0)])
    t = r.next
    r.gates += [("MulConstant", t, 1201, one), ("AssertZero", t)]
    r.next += 1
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("field", ["p101", "bls12_381"])
def test_gpu_assertion_order(field):
    p = FIELDS[field]
    r = order_relation(p)
    cases = [(), (1200,), (1201,), (0,), (MIN_CALLS - 1,), (100,), (5, 100), (1201, MIN_CALLS - 1), (1200, 0, 1201),
             (7, 900, 1201)]
    ws = []
    for nz in cases:
        w = [0] * r.n_wit
        for k in nz:
            w[k] = 1 + (k % 5)
        ws.append(w)
    msgs0 = r.messages(ws[0])
    b, e = record(0, msgs0)
    assert b.stats()["n_call_groups"] == 1 and b.stats()["n_asserts"] == 2 + 2 * MIN_CALLS
    b.finalize(True)
    v = b.evaluate(None, witness_array(r, ws), len(ws))
    for j, w in enumerate(ws):
        msgs = r.messages(w)
        expected = ev.evaluate(msgs)
        assert bool(v[j]["ok"]) == (expected == []), cases[j]
        # first failing sequence: before the loop 0, call c's k-th 1 + 2c + k, after the loop 1 + 2 * MIN_CALLS
        seqs = []
        if w[1200]:
            seqs.append(0)
        for c in range(MIN_CALLS):
            if w[c]:
                seqs.append(1 + 2 * c)
            if w[100]:
                seqs.append(1 + 2 * c + 1)
        if w[1201]:
            seqs.append(1 + 2 * MIN_CALLS)
        if seqs:
            assert int(v[j]["first_fail_seq"]) == min(seqs), cases[j]
        # the violation string from .sieve bytes
        b1, e1 = record(0, msgs)
        assert e1.get_violations() == expected, cases[j]


def run_batch(r, W, n_batch, no_groups, keep, wires, probe):
    b, e = record(0, r.messages(r.witness()), no_groups=no_groups)
    assert (b.stats()["n_call_groups"] == 0) == no_groups
    if keep:
        b.finalize(True)
    else:
        assert e.get_violations() is not None   # the Evaluator's own finalize: the live wires of its scope stay readable
    v = b.evaluate(None, W, n_batch)
    hs = [e.value_handle(x) for x in wires]
    vals = [b.read_values(j, hs, 32) for j in probe]
    return [(bool(x["ok"]), int(x["first_fail_seq"])) for x in v], vals


@pytest.mark.gpu
@pytest.mark.parametrize("n_batch", [1, 7, 64, 300])
@pytest.mark.parametrize("tile_log2", [None, "3"])
@pytest.mark.parametrize("keep", [0, 1])
def test_gpu_batches_grouped_equals_unrolled(n_batch, tile_log2, keep, monkeypatch):
    if tile_log2:
        monkeypatch.setenv("ZKB_TILE_LOG2", tile_log2)
    r = build(GOLDILOCKS if n_batch % 2 else BLS12_381_FR, 70, failing=True, n_asserts=1)
    rng = np.random.default_rng(n_batch)
    ws = [r.witness() for _ in range(n_batch)]
    W = witness_array(r, ws)
    wires = list(rng.choice(r.n_wit, 8, replace=False))    # witnesses and the loops' outputs: readable either way
    for first, count in r.blocks[1:]:
        wires += list(range(first, first + min(count, 6)))
    wires = [int(x) for x in wires]
    probe = sorted(set([0, n_batch - 1, n_batch // 2]))   # witness 0 is on a tile that is not resident when tiles > 1
    a = run_batch(r, W, n_batch, False, keep, wires, probe)
    s = run_batch(r, W, n_batch, True, keep, wires, probe)
    assert a[0] == s[0]
    assert a[1] == s[1]


@pytest.mark.gpu
def test_gpu_two_contexts_on_one_device():
    """zkb_evaluate_sharded over two contexts of device 0: the groups travel with the broadcast plan"""
    z = zkb()
    r = build(P127, 80, failing=True, n_asserts=2)
    buf = F.write_messages(r.messages(r.witness()))
    n_batch = 21
    ws = [r.witness() for _ in range(n_batch)]
    W = witness_array(r, ws)
    one = z.GpuBackend(0)
    e1 = z.Evaluator(one)
    e1.ingest_source(z.Source.from_buffers([buf]))
    assert one.stats()["n_call_groups"] >= 1
    one.finalize(keep_all_values=True)
    v_one = one.evaluate(None, W, n_batch)
    sh = z.ShardedBackend([0, 0])
    e = z.Evaluator(sh.root)
    e.ingest_source(z.Source.from_buffers([buf]))
    sh.root.finalize(keep_all_values=True)
    v = sh.evaluate(None, W, n_batch)
    assert (v["ok"] == v_one["ok"]).all() and (v["first_fail_seq"] == v_one["first_fail_seq"]).all()
    hs = [e.value_handle(x) for first, count in r.blocks for x in range(first, first + count, 37)]
    for j in (0, n_batch // 2, n_batch - 1):
        b, local = sh.owner(j, n_batch)
        assert b.read_values(local, hs, 32) == one.read_values(j, hs, 32), j
    sh.close()


@pytest.mark.gpu
def test_gpu_cli_evaluate_true_and_false(tmp_path):
    r = order_relation(BLS12_381_FR)
    for name, nz in (("true", ()), ("false", (MIN_CALLS - 1,))):
        w = [0] * r.n_wit
        for k in nz:
            w[k] = 3
        msgs = r.messages(w)
        expected = ev.evaluate(msgs)
        d = tmp_path / name
        d.mkdir()
        (d / "001_witness.sieve").write_bytes(F.write_messages(msgs[:1]))
        (d / "002_relation.sieve").write_bytes(F.write_messages(msgs[1:]))
        res = subprocess.run([CLI, "evaluate", str(d)], capture_output=True, text=True, timeout=300)
        if expected:
            assert res.returncode != 0
            assert "The statement is NOT TRUE!" in res.stderr
            assert f"- {expected[0]}" in res.stderr
        else:
            assert res.returncode == 0, res.stderr
            assert "The statement is TRUE!" in res.stderr
