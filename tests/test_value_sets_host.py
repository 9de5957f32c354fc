"""Value sets (zkb.h section 4) on a host-only context: one relation recorded once for many instance / witness sets.
Refusals, the recorded program (the same as a single statement of the longest streams), and each set's cut point (where
its own statement stops recording) against the oracle.  The device results are in tests/test_gpu_value_sets.py."""
import os
import subprocess

import numpy as np
import pytest

from oracle import evaluator as ev
from oracle import fixtures as fx
from oracle import ir
from oracle import sieve_fbs as F
from tests.gen_programs import Gen
from tests.util import ROOT, zkb

CLI = os.path.join(ROOT, "zkinterface-ir_b200", "zkb")
BLS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def buf(msgs):
    return F.write_messages(msgs)


def small_relation():
    h = fx.example_header()
    return h, ir.Relation(h, ir.ARITH, ir.SIMPLE, [], [
        ("Witness", 0), ("Instance", 1), ("Add", 2, 0, 1), ("AssertZero", 2),
        ("Witness", 3), ("Witness", 4), ("Mul", 5, 3, 4), ("AssertZero", 5)])


def wit(h, vals):
    return ir.Witness(h, [ir.literal32(v) for v in vals])


def host_evaluator():
    z = zkb()
    return z, z.Evaluator(z.GpuBackend(-1))


def test_refusals(tmp_path):
    h, rel = small_relation()
    z, e = host_evaluator()
    with pytest.raises(z.ZkbError) as err:   # no set yet
        e.get_batch_violations()
    assert err.value.code == z.ZKB_E_ARG
    with pytest.raises(z.ZkbError) as err:   # a relation inside a set
        e.add_value_set(z.Source.from_buffers([buf([wit(h, [1]), rel])]))
    assert err.value.code == z.ZKB_E_ARG and "Relation" in str(err.value)
    p = tmp_path / "s0"
    p.mkdir()
    (p / "001_witness.sieve").write_bytes(buf([wit(h, [1])]))
    (p / "002_relation.sieve").write_bytes(buf([rel]))
    with pytest.raises(z.ZkbError) as err:   # ... named by its file
        e.add_value_set(z.Source.from_directory(p))
    assert err.value.code == z.ZKB_E_ARG and "002_relation.sieve" in str(err.value)
    e.add_value_set(z.Source.from_buffers([buf([wit(h, [76, 0, 0])])]))
    e.ingest_source(z.Source.from_buffers([buf([fx.example_instance(), rel])]))
    with pytest.raises(z.ZkbError) as err:   # a set after a relation message
        e.add_value_set(z.Source.from_buffers([buf([wit(h, [1])])]))
    assert err.value.code == z.ZKB_E_ARG
    with pytest.raises(z.ZkbError) as err:   # common values after a relation message
        e.ingest_source(z.Source.from_buffers([buf([wit(h, [1])])]))
    assert err.value.code == z.ZKB_E_ARG
    for call in (e.get_violations, lambda: e.get(2)):
        with pytest.raises(z.ZkbError) as err:
            call()
        assert err.value.code == z.ZKB_E_ARG
    for bad in (1, 7):
        with pytest.raises(z.ZkbError) as err:
            e.value_set_cut(bad)
        assert err.value.code == z.ZKB_E_ARG and "out of range" in str(err.value)
    with pytest.raises(z.ZkbError) as err:
        e.get_of(1, 2)
    assert err.value.code == z.ZKB_E_ARG
    with pytest.raises(z.ZkbError) as err:   # host-only: recording works, results need the device
        e.get_batch_violations()
    assert err.value.code == z.ZKB_E_CUDA
    # flatten / expand-definable evaluators take no value set, and a batch evaluator cannot become one
    for kw in ({"flatten": True}, {"expand_gate_set": "arithmetic"}):
        f = z.Evaluator(**kw)
        with pytest.raises(z.ZkbError) as err:
            f.add_value_set(z.Source.from_buffers([buf([wit(h, [1])])]))
        assert err.value.code == z.ZKB_E_ARG
    g = z.Evaluator(z.GpuBackend(-1))
    g.add_value_set(z.Source.from_buffers([buf([wit(h, [1])])]))
    with pytest.raises(z.ZkbError) as err:
        g._chk(z._lib.zkb_evaluator_set_flatten(g._e, 1))
    assert err.value.code == z.ZKB_E_ARG


def test_use_devices_refusals():
    z, e = host_evaluator()
    other = z.GpuBackend(-1)
    for ctxs in ([other], [e.backend, other], [e.backend]):   # not the backend first / not a communicator
        import ctypes as C
        arr = (C.c_void_p * len(ctxs))(*[b._c for b in ctxs])
        rc = z._lib.zkb_evaluator_use_devices(e._e, arr, len(ctxs))
        assert rc == z.ZKB_E_ARG
        assert "use_devices" in z._lib.zkb_evaluator_last_error(e._e).decode()


def streams(msgs):
    inst, wit, rel = msgs
    return list(inst.common_inputs), list(wit.short_witness), rel


def make_sets(seed, msgs, n_sets):
    """(common instance, common witness, [(instance, witness)] per set) from a statement's streams: random splits, lengths
    from short to longer than the relation consumes, and random values"""
    rng = np.random.default_rng(seed)
    inst, wv, rel = streams(msgs)
    ci = int(rng.integers(0, len(inst) + 1)) if rng.random() < 0.4 else 0
    cw = int(rng.integers(0, len(wv) + 1)) if rng.random() < 0.4 else 0
    h = rel.header
    p = int.from_bytes(h.field_characteristic, "little")

    def rand_vals(n):
        return [ir.le_bytes(int(rng.integers(0, min(p, 1 << 62)))) for _ in range(n)]

    sets = []
    for j in range(n_sets):
        ni = max(0, len(inst) - ci + int(rng.integers(-3, 3)))
        nw = max(0, len(wv) - cw + int(rng.integers(-4, 3)))
        if j == 0:
            ni, nw = len(inst) - ci, len(wv) - cw
        si = (inst[ci:] + rand_vals(max(0, ni - (len(inst) - ci))))[:ni]
        sw = (wv[cw:] + rand_vals(max(0, nw - (len(wv) - cw))))[:nw]
        sets.append((si, sw))
    return inst[:ci], wv[:cw], sets


def set_statement(h, common, s, rel):
    ci, cw = common
    si, sw = s
    return [ir.Instance(h, ci), ir.Instance(h, si), ir.Witness(h, cw), ir.Witness(h, sw), rel]


def record_batch(z, h, common_i, common_w, sets, rel, backend=None):
    e = z.Evaluator(backend or z.GpuBackend(-1))
    for si, sw in sets:
        e.add_value_set(z.Source.from_buffers([buf([ir.Instance(h, si), ir.Witness(h, sw)])]))
    e.ingest_source(z.Source.from_buffers([buf([ir.Instance(h, common_i), ir.Witness(h, common_w), rel])]))
    return e


class NoFailTracing(ev.TracingBackend):
    """records every assertion and lets it pass: the oracle then stops only where the streams (or the relation) stop it"""

    def assert_zero(self, w):
        self.asserts.append((len(self.trace), w[0], w[1] == 0))


def oracle_cut(msgs):
    """(kind, seq) where the oracle stops recording this statement: kind 'instance' / 'witness' / 'error' / None"""
    tb = NoFailTracing()
    try:
        o = ev.Evaluator.from_messages(msgs, tb)
        viol = o.get_violations()
    except ir.OraclePanic as p:
        return ("witness" if "Missing witness value" in str(p) else "error"), len(tb.asserts)
    errs = [v for v in viol if v != "Did not receive any gate to verify."]
    if not errs:
        return None, None
    return ("instance" if errs[0] == "Not enough instance to consume" else "error"), len(tb.asserts)


CASES = [(seed, 101, False) for seed in range(20)] + [(seed, 2, True) for seed in range(100, 110)] + \
        [(seed, (1 << 64) - (1 << 32) + 1, False) for seed in range(200, 204)] + [(300, BLS, False)]


@pytest.mark.parametrize("seed,p,boolean", CASES)
def test_cut_points_match_the_oracle(seed, p, boolean):
    z = zkb()
    msgs = Gen(seed, p, boolean).statement()
    h = msgs[2].header
    ci, cw, sets = make_sets(seed, msgs, 12)
    e = record_batch(z, h, ci, cw, sets, msgs[2])
    for j, s in enumerate(sets):
        kind, seq = oracle_cut(set_statement(h, (ci, cw), s, msgs[2]))
        what, got = e.value_set_cut(j)
        want = {None: (0,), "instance": (1, 3), "witness": (2, 3), "error": (3,)}[kind]
        assert what in want and got == seq, (j, kind, seq, what, got)


@pytest.mark.parametrize("n_wit,want", [(0, (2, 1)), (1, (2, 2)), (2, (2, 3)), (3, (2, 3)), (4, (0, None))])
def test_cut_inside_switch_branches(n_wit, want):
    """case 0 consumes one witness value, case 1 three: a set with one or two values runs out inside the second branch"""
    z = zkb()
    h = fx.example_header()
    zero = ir.literal32(0)
    rel = ir.Relation(h, ir.ARITH, ir.FOR_FUNCTION_SWITCH, [], [
        ("Instance", 0), ("AssertZero", 0),
        ("Switch", 0, [], [bytes([0]), bytes([1])], [
                ("AbstractAnonCall", [], 0, 1, [("Witness", 1), ("AssertZero", 1)]),
            ("AbstractAnonCall", [], 0, 3, [("Witness", 1), ("Witness", 2), ("AssertZero", 2), ("Witness", 3), ("Add", 4, 1, 3)])]),
        ("Witness", 5), ("AssertZero", 5)])
    sets = [([zero], [zero] * 4), ([zero], [zero] * n_wit)]
    e = record_batch(z, h, [], [], sets, rel)
    kind, seq = oracle_cut(set_statement(h, ([], []), sets[1], rel))
    assert e.value_set_cut(1) == want
    assert (kind, seq) == ({2: "witness", 0: None}[want[0]], want[1])


@pytest.mark.parametrize("seed,p,boolean", CASES[::3])
def test_batch_records_the_program_of_the_longest_streams(seed, p, boolean):
    z = zkb()
    msgs = Gen(seed, p, boolean).statement()
    h = msgs[2].header
    ci, cw, sets = make_sets(seed + 7, msgs, 9)
    e = record_batch(z, h, ci, cw, sets, msgs[2])
    li = max((s[0] for s in sets), key=len)
    lw = max((s[1] for s in sets), key=len)
    b1 = z.GpuBackend(-1)
    one = z.Evaluator(b1)
    one.ingest_source(z.Source.from_buffers([buf([ir.Instance(h, ci + li), ir.Witness(h, cw + lw), msgs[2]])]))
    k0, a0, c0 = e.backend.program()
    k1, a1, c1 = b1.program()
    assert np.array_equal(k0, k1) and np.array_equal(a0, a1) and np.array_equal(c0, c1)
    s0, s1 = e.backend.stats(), b1.stats()
    for key in ("n_values", "n_asserts", "n_instance", "n_witness", "n_consts", "ir_gates", "callbacks", "n_call_groups"):
        assert s0[key] == s1[key], key
    assert e.backend.pending_error() == b1.pending_error()


def test_common_values_and_raw_values_keep_their_positions():
    """common instance values come first in every set's stream; set positions follow them"""
    z = zkb()
    h, rel = small_relation()
    e = record_batch(z, h, [ir.literal32(25)], [ir.literal32(3)], [([], [ir.literal32(7), ir.literal32(101 + 5)])], rel)
    k, a, b = e.backend.program()
    assert [int(x) for x, kk in zip(b, k) if kk == 2] == [0, 1, 2]
    assert e.value_set_cut(0) == (0, None)


def cli(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, timeout=60)


def test_cli_usage_errors(tmp_path):
    (tmp_path / "sets").mkdir()
    for args in (["evaluate", "--devices", "0,0", str(tmp_path)],                               # --devices without --sets
                 ["evaluate", "--device", "0", "--devices", "0", "--sets", str(tmp_path / "sets"), str(tmp_path)],
                 ["evaluate", "--devices", "0,x", "--sets", str(tmp_path / "sets"), str(tmp_path)],
                 ["evaluate", "--devices", "", "--sets", str(tmp_path / "sets"), str(tmp_path)]):
        r = cli(*args)
        assert r.returncode == 2 and r.stderr.startswith("usage:"), args
    r = cli("evaluate", "--sets", str(tmp_path / "missing"), str(tmp_path))
    assert r.returncode == 1 and "Error: cannot read directory" in r.stderr
