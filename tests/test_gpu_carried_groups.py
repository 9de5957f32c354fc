"""Carried loops over prime fields on the device (kernels.cu: k_arith_chain): values and verdicts against
oracle/evaluator.py, and bit-for-bit parity with the gate-by-gate recording (ZKB_NO_CALL_GROUPS=1) over batches, tiles,
read-back, capture, a long chain, sharded and broadcast contexts and `zkb evaluate --sets`."""
import os
import subprocess

import numpy as np
import pytest

from oracle import evaluator as ev
from oracle import ir
from oracle import sieve_fbs as F
from tests.test_arith_call_groups_host import BLS12_381_FR, FIELDS, GOLDILOCKS, MIN_CALLS, P127, C, I, add, mul, record
from tests.test_carried_groups_host import WIDE, ChainRel, build_chains, chain_then_group
from tests.util import zkb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "zkinterface-ir_b200", "zkb")


def witness_array(r, ws):
    return np.array([[list(r.le(x % (1 << (8 * r.nb)))) for x in w] for w in ws], dtype=np.uint8)


def readable_wires(r):
    """a few wires of every block (witnesses, instances, group and chain outputs) and the tail's sums"""
    wires = []
    for first, count in r.blocks:
        wires += list(range(first, first + count, max(1, count // 7)))
    return sorted(set(wires))


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(WIDE))
@pytest.mark.parametrize("seed", [0, 1])
def test_gpu_chain_values_and_verdicts(field, seed):
    r, n_chains = build_chains(FIELDS[field], seed, n_asserts=1)
    inst = r.instance_values()
    msgs = r.messages(r.witness(), inst)
    expected = ev.evaluate(msgs)
    b, e = record(0, msgs)
    assert b.stats()["n_carried_groups"] == n_chains
    b.finalize(True)
    assert e.get_violations() == expected
    if expected == []:
        o = ev.Evaluator.from_messages(msgs, ev.PlaintextBackend())
        for wid, val in o.values.items():
            assert e.get(wid) == val, wid


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(WIDE))
def test_gpu_raw_values_as_seeds_and_inputs(field):
    """witness values >= p (kept unreduced by the reference) as seeds and as non-carried inputs"""
    r, _ = build_chains(FIELDS[field], 50, n_asserts=1, raw=True)
    w = r.witness()
    assert any(x >= r.p for x in w)
    msgs = r.messages(w)
    b, e = record(0, msgs)
    assert e.get_violations() == ev.evaluate(msgs)
    bs, es = record(0, msgs, no_groups=True)
    assert es.get_violations() == e.get_violations()
    hs, hu = [e.value_handle(x) for x in readable_wires(r)], [es.value_handle(x) for x in readable_wires(r)]
    assert b.read_values(0, hs, 32) == bs.read_values(0, hu, 32)


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(WIDE))
def test_gpu_group_reading_a_chain(field):
    """depth order and callout slots: a chain seeded by a group's outputs, a group that reads the chain's outputs"""
    r = chain_then_group(FIELDS[field])
    msgs = r.messages(r.witness())
    b, e = record(0, msgs)
    assert b.stats()["n_carried_groups"] == 1 and b.stats()["n_call_groups"] == 3
    b.finalize(True)
    assert e.get_violations() == ev.evaluate(msgs) == []
    o = ev.Evaluator.from_messages(msgs, ev.PlaintextBackend())
    for wid, val in o.values.items():
        assert e.get(wid) == val, wid


def horner_check(p, n_calls):
    """acc = acc * x + c_i (x and c_i witnesses), a grand product g = g * a_i over an anonymous body checked against
    witnesses b_i with one AssertZero per step, and gates after the loops that read the chains' last outputs.  Witness
    layout: c_i, a_i, b_i (n each), x, then the two seeds (3n + 1, 3n + 2)."""
    r = ChainRel(p, 3, n_wit=3 * n_calls + 1)
    m1 = r.le(p - 1)
    r.funcs.append(ir.Function("horner", 1, 3, 0, 0, [("Mul", 4, 1, 2), ("Add", 0, 4, 3)]))
    prod = [("Mul", 0, 1, 2), ("MulConstant", 4, 3, m1), ("Add", 5, 0, 4), ("AssertZero", 5)]
    r.witnesses()
    x = 3 * n_calls
    hb, _ = r.chain(("horner", 1, 3, "plain"), [("carry", 0, 1), ("aff", x, 0), ("aff", 0, 1)], n_calls=n_calls, seeds=["witness"],
                    S_extra=0)
    gb, _ = r.chain(("prod", 1, 3, "plain"), [("carry", 0, 1), ("aff", n_calls, 1), ("aff", 2 * n_calls, 1)], n_calls=n_calls,
                    seeds=["witness"], S_extra=0, anon_body=prod)
    s = r.next
    r.gates += [("Add", s, hb + n_calls - 1, gb + n_calls - 1), ("MulConstant", s + 1, s, r.le(1))]
    r.next += 2
    return r, hb, gb


def horner_witness(r, n, corrupt=None):
    """corrupt: the step whose b_i is off by one"""
    p = r.p
    rng = np.random.default_rng(n + (corrupt or 0))
    c = [int(v) for v in rng.integers(0, 1 << 62, n)]
    a = [int(v) for v in rng.integers(1, 1 << 62, n)]
    x, h0, g0 = (int(v) for v in rng.integers(1, 1 << 62, 3))
    b, g = [], g0
    for i in range(n):
        g = g * a[i] % p
        b.append(g)
    if corrupt is not None:
        b[corrupt] = (b[corrupt] + 1) % p
    return c + a + b + [x, h0, g0]


@pytest.mark.gpu
@pytest.mark.parametrize("field", list(WIDE))
def test_gpu_failing_step_mid_chain(field):
    """a corrupted b_i fails step i's assertion: the same first failure and violation text as unrolled and the oracle"""
    n = MIN_CALLS + 5
    r, _, _ = horner_check(FIELDS[field], n)
    for corrupt in (None, 0, 700, n - 1):
        msgs = r.messages(horner_witness(r, n, corrupt))
        b, e = record(0, msgs)
        assert b.stats()["n_carried_groups"] == 2
        bs, es = record(0, msgs, no_groups=True)
        assert e.get_violations() == es.get_violations() == ev.evaluate(msgs), corrupt
        assert (e.get_violations() == []) == (corrupt is None)


def run_batch(r, W, n_batch, no_groups, keep, wires, probe):
    b, e = record(0, r.messages(W[0]), no_groups=no_groups)
    assert (b.stats()["n_carried_groups"] == 0) == no_groups
    if keep:
        b.finalize(True)
    else:
        assert e.get_violations() is not None
    Wa = witness_array(r, W)
    v = b.evaluate(None, Wa, n_batch)
    hs = [e.value_handle(x) for x in wires]
    vals = [b.read_values(j, hs, 32) for j in probe]
    b.capture(hs)
    v2 = b.evaluate(None, Wa, n_batch)
    cap = b.read_captured(0, n_batch, 32)
    return [(bool(x["ok"]), int(x["first_fail_seq"])) for x in v], vals, [(bool(x["ok"]), int(x["first_fail_seq"])) for x in v2], cap


@pytest.mark.gpu
@pytest.mark.parametrize("n_batch", [1, 7, 64, 300])
@pytest.mark.parametrize("tile_log2", [None, "3"])
@pytest.mark.parametrize("keep", [0, 1])
def test_gpu_batches_grouped_equals_unrolled(n_batch, tile_log2, keep, monkeypatch):
    if tile_log2:
        monkeypatch.setenv("ZKB_TILE_LOG2", tile_log2)
    p = P127 if n_batch % 2 else BLS12_381_FR
    n = MIN_CALLS + 3
    r, hb, gb = horner_check(p, n)
    ws = [horner_witness(r, n, None if j % 3 else (j * 37) % n) for j in range(n_batch)]
    wires = [hb, hb + 1, hb + n - 1, gb, gb + n // 2, gb + n - 1, r.next - 1, 0, 3 * n]
    probe = sorted(set([0, n_batch - 1, n_batch // 2]))
    a = run_batch(r, ws, n_batch, False, keep, wires, probe)
    s = run_batch(r, ws, n_batch, True, keep, wires, probe)
    assert a[0] == s[0] and a[2] == s[2] == a[0]
    assert a[1] == s[1]
    assert np.array_equal(a[3], s[3])
    for j in range(n_batch):
        assert a[0][j][0] == (j % 3 != 0), j


@pytest.mark.gpu
def test_gpu_long_chain_grouped_equals_unrolled():
    n = 1 << 16
    r, hb, gb = horner_check(BLS12_381_FR, n)
    w = horner_witness(r, n)
    msgs = r.messages(w)
    b, e = record(0, msgs)
    bs, es = record(0, msgs, no_groups=True)
    assert b.stats()["n_carried_groups"] == 2
    assert e.get_violations() == es.get_violations() == []
    wires = [hb, hb + n // 3, hb + n - 1, gb + n - 1, r.next - 1]
    assert b.read_values(0, [e.value_handle(x) for x in wires], 32) == bs.read_values(0, [es.value_handle(x) for x in wires], 32)
    p = r.p
    acc = w[3 * n + 1]
    for i in range(n):
        acc = (acc * w[3 * n] + w[i]) % p
    assert e.get(hb + n - 1) == acc


@pytest.mark.gpu
def test_gpu_sharded_and_broadcast():
    """zkb_evaluate_sharded over two contexts of device 0: the chains travel with the broadcast plan"""
    z = zkb()
    n = MIN_CALLS + 1
    r, hb, gb = horner_check(P127, n)
    n_batch = 21
    ws = [horner_witness(r, n, None if j % 4 else j) for j in range(n_batch)]
    buf = F.write_messages(r.messages(ws[0]))
    W = witness_array(r, ws)
    one = z.GpuBackend(0)
    e1 = z.Evaluator(one)
    e1.ingest_source(z.Source.from_buffers([buf]))
    assert one.stats()["n_carried_groups"] == 2
    one.finalize(keep_all_values=True)
    v_one = one.evaluate(None, W, n_batch)
    sh = z.ShardedBackend([0, 0])
    e = z.Evaluator(sh.root)
    e.ingest_source(z.Source.from_buffers([buf]))
    sh.root.finalize(keep_all_values=True)
    assert sh.root.plan_hash() == one.plan_hash()
    v = sh.evaluate(None, W, n_batch)
    assert (v["ok"] == v_one["ok"]).all() and (v["first_fail_seq"] == v_one["first_fail_seq"]).all()
    assert sh.backends[1].stats()["n_carried_groups"] == 2
    hs = [e.value_handle(x) for x in (hb, hb + n - 1, gb + 5, r.next - 1)]
    for j in (0, n_batch // 2, n_batch - 1):
        b, local = sh.owner(j, n_batch)
        assert b.read_values(local, hs, 32) == one.read_values(j, hs, 32), j
    sh.close()


@pytest.mark.gpu
def test_gpu_cli_evaluate_sets(tmp_path):
    """one relation, two witness sets (the second fails mid-chain): each set's verdict as `zkb evaluate` prints it"""
    n = MIN_CALLS
    r, _, _ = horner_check(BLS12_381_FR, n)
    ws = [horner_witness(r, n), horner_witness(r, n, 17)]
    (tmp_path / "relation.sieve").write_bytes(F.write_messages(r.messages(ws[0])[1:]))
    sets = tmp_path / "sets"
    for k, w in enumerate(ws):
        (sets / f"s{k}").mkdir(parents=True)
        (sets / f"s{k}" / "witness.sieve").write_bytes(F.write_messages(r.messages(w)[:1]))
    expected = [ev.evaluate(r.messages(w)) for w in ws]
    assert expected[0] == [] and expected[1] != []
    res = subprocess.run([CLI, "evaluate", "--sets", str(sets), str(tmp_path / "relation.sieve")], capture_output=True, text=True,
                         timeout=300)
    out = res.stdout + res.stderr
    assert res.returncode != 0
    s0, s1 = out.index("== s0 =="), out.index("== s1 ==")
    assert "The statement is TRUE!" in out[s0:s1]
    assert "The statement is NOT TRUE!" in out[s1:] and f"- {expected[1][0]}" in out[s1:]
