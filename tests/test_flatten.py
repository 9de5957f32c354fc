"""`flatten` (cli.rs:442-472): the C++ Evaluator in flatten mode + the C++ FlatBuffers writer must emit, gate for
gate and value for value, what the reference's IRFlattener emits (restated in oracle/flattening.py), and the
flattened statement must evaluate like the original (flattening.rs:200-252)."""
import os

import pytest

from oracle import evaluator as ev
from oracle import fixtures as fx
from oracle import flattening as fl
from oracle import ir
from oracle import sieve_fbs as F
from tests.test_host_evaluator import STATEMENTS
from tests.util import zkb


def oracle_flatten(msgs):
    f = fl.IRFlattener()
    e = ev.Evaluator.from_messages(msgs, f)
    return f.finish(), e


def ours_flatten(msgs):
    z = zkb()
    e = z.Evaluator(flatten=True)
    e.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
    return e, e.flatten()


def test_oracle_flattener_pinned_on_reference_tests():
    # flattening.rs:200-252: flatten(example) validates (checked in test_validator.py) and evaluates to no violation
    msgs = [fx.example_instance(), fx.example_witness(), fx.example_relation()]
    flat, _ = oracle_flatten(msgs)
    assert ev.evaluate(flat) == []
    rel = [m for m in flat if isinstance(m, ir.Relation)]
    assert len(rel) == 1 and rel[0].feat_mask == ir.SIMPLE and rel[0].gate_mask == ir.ARITH
    # one gate per ZKBackend callback: 283 for the example (SURVEY.md 8c)
    assert len(rel[0].gates) == 283
    # the incorrect witness still flattens completely (the flattener does not evaluate) and then fails
    bad, _ = oracle_flatten([fx.example_instance(), fx.example_witness_incorrect(), fx.example_relation()])
    assert len([m for m in bad if isinstance(m, ir.Relation)][0].gates) == 283
    v = ev.evaluate(bad)
    assert len(v) == 1 and v[0].startswith("Wire_") and v[0].endswith("should be 0, while it is not")


@pytest.mark.parametrize("name", list(STATEMENTS))
def test_flatten_matches_the_reference_flattener(name):
    msgs = STATEMENTS[name]()
    want, _ = oracle_flatten(msgs)
    e, (ib, wb, rb) = ours_flatten(msgs)
    got = F.read_messages(ib) + F.read_messages(wb) + F.read_messages(rb)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert type(g) is type(w)
        assert g.header.field_characteristic == w.header.field_characteristic
        assert g.header.version == w.header.version and g.header.field_degree == w.header.field_degree
        if isinstance(w, ir.Relation):
            assert (g.gate_mask, g.feat_mask, g.functions) == (w.gate_mask, w.feat_mask, [])
            assert g.gates == w.gates
        elif isinstance(w, ir.Instance):
            assert g.common_inputs == w.common_inputs
        else:
            assert g.short_witness == w.short_witness
    # the flattened statement has the same verdict as the original
    assert ev.evaluate(got) == ev.evaluate(msgs) == []
    # and our own reader takes what our writer wrote: same callbacks minus nothing (copies are gates now)
    z = zkb()
    b2 = z.GpuBackend(-1)
    e2 = z.Evaluator(b2)
    e2.ingest_source(z.Source.from_buffers([ib, wb, rb]))
    assert b2.pending_error() is None
    assert sum(b2.stats()["callbacks"].values()) >= len([m for m in want if isinstance(m, ir.Relation)][0].gates)


def test_flatten_cuts_messages_every_100000(tmp_path):
    # builder.rs:69,93-98: a 250 001-gate relation leaves as 3 messages; values likewise
    h = fx.example_header()
    n = 250_000
    gates = [("Witness", 0)] + [("Add", i + 1, i, i) for i in range(n)]
    rel = ir.Relation(h, ir.ARITH, ir.SIMPLE, [], gates)
    msgs = [ir.Witness(h, [b"\x01"]), rel]
    z = zkb()
    e = z.Evaluator(flatten=True)
    e.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
    e.flatten_to_dir(tmp_path / "out" / "deep")
    names = sorted(os.listdir(tmp_path / "out" / "deep"))
    assert names == ["000_instance.sieve", "001_witness.sieve", "002_relation.sieve"]
    rb = (tmp_path / "out" / "deep" / "002_relation.sieve").read_bytes()
    parts = F.split_messages(rb)
    assert len(parts) == 3
    assert (tmp_path / "out" / "deep" / "000_instance.sieve").read_bytes() == b""
    sizes = [len(F.read_message(p).gates) for p in parts]
    assert sizes == [100_000, 100_000, 50_001]
    # bytes per simple gate with shared vtables (3 Wire tables of 16 B, gate table 16 B, Directive 12 B, vector slot 4 B)
    assert len(rb) / (n + 1) < 84
    # a second flatten into the same directory replaces the files (FilesSink::new_clean)
    e.flatten_to_dir(tmp_path / "out" / "deep")
    assert (tmp_path / "out" / "deep" / "002_relation.sieve").read_bytes() == rb
    # multi-message buffers go through the parallel parser: same program either way
    b1, b2 = z.GpuBackend(-1), z.GpuBackend(-1)
    e1, e2 = z.Evaluator(b1), z.Evaluator(b2)
    wbuf = F.write_message(msgs[0])
    e1.ingest_source(z.Source.from_buffers([wbuf, rb]))
    e2.ingest_message(wbuf)
    for p in parts:
        e2.ingest_message(p)
    k1, a1, bb1 = b1.program()
    k2, a2, bb2 = b2.program()
    assert (k1 == k2).all() and (a1 == a2).all() and (bb1 == bb2).all() and len(k1) == n + 1


def test_flatten_mode_refuses_evaluation(tmp_path):
    z = zkb()
    msgs = STATEMENTS["example"]()
    e, _ = ours_flatten(msgs)
    with pytest.raises(z.ZkbError):
        e.get_violations()
    with pytest.raises(z.ZkbError):
        e.flatten_to_dir(str(tmp_path / "x.sieve"))


@pytest.mark.parametrize("name", list(STATEMENTS))
def test_writer_round_trips_every_message_kind(name):
    """C++ reader -> owned structs -> C++ writer -> oracle reader == oracle reader of the original (For / Switch /
    Call / AnonCall / functions / iterator expressions included)"""
    z = zkb()
    b = z.GpuBackend(-1)
    for m in STATEMENTS[name]():
        raw = F.write_message(m)
        again = b.rewrite_message(raw)
        assert again[8:12] == b"siev" and int.from_bytes(again[:4], "little") == len(again) - 4
        assert F.read_message(again) == F.read_message(raw)
        # and it is a fixed point of our own reader/writer pair
        assert b.rewrite_message(again) == again


def test_writer_round_trips_the_reference_binary_fixtures():
    import glob
    z = zkb()
    b = z.GpuBackend(-1)
    golden = os.path.join(os.path.dirname(__file__), "golden")
    n = 0
    for path in sorted(glob.glob(os.path.join(golden, "**", "*.sieve"), recursive=True)):
        for raw in F.split_messages(open(path, "rb").read()):
            assert F.read_message(b.rewrite_message(raw)) == F.read_message(raw), path
            n += 1
    assert n >= 9


# ---- ExpandDefinable (consumers/exp_definable.rs) in front of the flattener ---------------------------------
EXPAND_CASES = [
    ("example", "@add,@mul"),                  # AddConstant / MulConstant become Constant + Add / Mul
    ("example", "arithmetic"),                 # nothing to rewrite
    ("builder_switch", "@add,@mul,@mulc"),
    ("boolean", "@add,@mul"),                  # And -> Mul, Xor -> Add, Not -> Constant(1) + Add
    ("boolean", "@xor,@and,@addc"),            # Not needs ADD: panic
    ("example", "@xor,@and"),                  # Add -> Xor, Mul -> And (nonsense over p = 101, but that is what it does)
    ("example", "@mul"),                       # Add cannot be replaced: panic
]


@pytest.mark.parametrize("name,gate_set", EXPAND_CASES)
def test_expand_definable_matches_the_reference(name, gate_set):
    z = zkb()
    msgs = STATEMENTS[name]()
    mask = ir.parse_gate_set(gate_set) if hasattr(ir, "parse_gate_set") else None
    if mask is None:
        bits = {"@add": ir.ADD, "@addc": ir.ADDC, "@mul": ir.MUL, "@mulc": ir.MULC, "@xor": ir.XOR, "@and": ir.AND, "@not": ir.NOT,
                "arithmetic": ir.ARITH, "boolean": ir.BOOL}
        mask = 0
        for tok in gate_set.split(","):
            mask |= bits[tok]
    x = fl.ExpandDefinable(mask)
    panic = None
    try:
        ev.Evaluator.from_messages(msgs, x)
    except ir.OraclePanic as e:
        panic = str(e)
    e = z.Evaluator(expand_gate_set=gate_set)
    if panic is not None:
        with pytest.raises(z.ZkbError) as err:
            e.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
        assert err.value.code == z.ZKB_E_FATAL and str(err.value) == panic
        return
    want = x.finish()
    e.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
    ib, wb, rb = e.flatten()
    got = F.read_messages(ib) + F.read_messages(wb) + F.read_messages(rb)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert type(g) is type(w)
        if isinstance(w, ir.Relation):
            assert g.gates == w.gates and g.gate_mask == w.gate_mask
        elif isinstance(w, ir.Instance):
            assert g.common_inputs == w.common_inputs
        else:
            assert g.short_witness == w.short_witness
    allowed = {"Constant", "AssertZero", "Copy", "Instance", "Witness"}
    names = {"@add": "Add", "@addc": "AddConstant", "@mul": "Mul", "@mulc": "MulConstant", "@xor": "Xor", "@and": "And", "@not": "Not"}
    if gate_set == "arithmetic":
        allowed |= {"Add", "AddConstant", "Mul", "MulConstant"}
    else:
        allowed |= {names[t] for t in gate_set.split(",")}
    for m in got:
        if isinstance(m, ir.Relation):
            assert {g[0] for g in m.gates} <= allowed
    if gate_set in ("@add,@mul", "arithmetic", "@add,@mul,@mulc"):
        assert ev.evaluate(got) == ev.evaluate(msgs) == []      # the rewritten statement means the same


def test_expand_definable_gate_set_errors_and_cli(tmp_path):
    import subprocess
    z = zkb()
    with pytest.raises(z.ZkbError) as err:
        z.Evaluator(expand_gate_set="@nope")
    assert "Unable to parse the following gateset" in str(err.value)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "zkinterface-ir_b200", "zkb")
    out = tmp_path / "expanded"
    r = subprocess.run([cli, "expand-definable", "--gate-set", "@add,@mul", "--out", str(out),
                        os.path.join(root, "tests", "golden", "example")], capture_output=True, timeout=60)
    assert r.returncode == 0, r.stderr
    msgs = [m for n in sorted(os.listdir(out)) for m in F.read_messages((out / n).read_bytes())]
    kinds = {g[0] for m in msgs if isinstance(m, ir.Relation) for g in m.gates}
    assert "AddConstant" not in kinds and "MulConstant" not in kinds and ev.evaluate(msgs) == []


def test_flatten_without_a_witness_like_the_verifier():
    """the IRFlattener takes witness(None) (flattening.rs:178-190): flattening a relation without a witness file emits the
    Witness gates and no witness message; the evaluating backend would have panicked instead"""
    z = zkb()
    msgs = [fx.example_instance(), fx.example_relation()]
    want, _ = oracle_flatten(msgs)
    e, (ib, wb, rb) = ours_flatten(msgs)
    assert wb == b""
    got = F.read_messages(ib) + F.read_messages(rb)
    assert [type(m) for m in got] == [type(m) for m in want]
    assert got[-1].gates == want[-1].gates and got[0].common_inputs == want[0].common_inputs
    assert sum(1 for g in got[-1].gates if g[0] == "Witness") > 0
    with pytest.raises(z.ZkbError) as err:                      # not in flatten mode: PlaintextBackend::witness(None) panics
        ev2 = z.Evaluator(z.GpuBackend(-1))
        ev2.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
    assert err.value.code == z.ZKB_E_FATAL and str(err.value) == "Missing witness value for PlaintextBackend"
