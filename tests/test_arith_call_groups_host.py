"""Loop-structured recording over prime fields (csrc/program.h CallGroup, evaluator.cpp arith_template_of): a For loop of at
least kArithGroupMinCalls = 1024 calls of a plain named function whose body holds Constant / Add / Mul / AddConstant /
MulConstant gates and AssertZero on computed wires is kept as ONE descriptor.  Everything the gate-by-gate unrolling
(rust/src/consumers/evaluator.rs:495-559 + :441-471 + :698-746) makes observable must stay the same: callback counts,
ir_gates, assertion count and source wires, scope bindings, pending errors.  Host-only contexts (no GPU)."""
import os

import numpy as np
import pytest

from oracle import evaluator as ev
from oracle import ir
from oracle import sieve_fbs as F
from tests.util import zkb

I = lambda n: ("Name", n)
C = lambda v: ("Const", v)
add = lambda l, r: ("Add", l, r)
mul = lambda l, r: ("Mul", l, r)

P101 = 101
GOLDILOCKS = 2**64 - 2**32 + 1
P127 = 2**127 - 1
BLS12_381_FR = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
FIELDS = {"p101": P101, "goldilocks": GOLDILOCKS, "p127": P127, "bls12_381": BLS12_381_FR}
MIN_CALLS = 1024


class ArithRel:
    """random prime-field relation: a block of witnesses, plain functions, For loops of >= 1024 calls over them, a tail"""

    def __init__(self, p, seed, n_wit=1100, raw_witness=False):
        self.p = p
        self.nb = (p.bit_length() + 7) // 8
        self.rng = np.random.default_rng(seed)
        self.h = ir.Header(p.to_bytes(self.nb, "little"))
        self.n_wit = n_wit
        self.raw = raw_witness
        self.funcs, self.gates, self.blocks = [], [], []
        self.next = 0

    def ri(self, lo, hi):
        return int(self.rng.integers(lo, hi + 1))

    def rval(self, lo, hi):
        """uniform integer in [lo, hi) for any width"""
        span = hi - lo
        nbytes = (span.bit_length() + 7) // 8 + 8
        return lo + int.from_bytes(self.rng.bytes(nbytes), "little") % span

    def le(self, v):
        return int(v).to_bytes(self.nb, "little")

    def const(self, ge_p=False):
        return self.le(self.rval(self.p, 1 << (8 * self.nb)) if ge_p else self.rval(0, self.p))

    def function(self, name, n_out, n_in, kind="plain", n_asserts=0):
        """kind 'plain' qualifies (with n_asserts always-true AssertZero gates on computed wires); the others must be
        refused and run gate by gate: 'and' / 'xor' / 'not' / 'copy' in the body, 'assert_input', 'raw_const'"""
        g, avail = [], list(range(n_out, n_out + n_in))
        nxt = n_out + n_in
        n_body = self.ri(max(n_out, 2), 12)
        targets = [None] * (n_body - n_out) + list(range(n_out))
        computed = []
        for t in targets:
            w = t if t is not None else nxt
            if t is None:
                nxt += 1
            op = ["Add", "Mul", "AddConstant", "MulConstant", "Constant"][self.ri(0, 4)]
            a, b = avail[self.ri(0, len(avail) - 1)], avail[self.ri(0, len(avail) - 1)]
            if op in ("Add", "Mul"):
                g.append((op, w, a, b))
            elif op in ("AddConstant", "MulConstant"):
                g.append((op, w, a, self.const(ge_p=self.ri(0, 5) == 0)))   # reduced result: a constant >= p is fine
            else:
                g.append((op, w, self.const()))
            avail.append(w)
            computed.append(w)
        for k in range(n_asserts):      # x - x for a computed x: zero on every witness
            x = computed[self.ri(0, len(computed) - 1)]
            g.append(("MulConstant", nxt, x, self.le(self.p - 1)))
            g.append(("Add", nxt + 1, x, nxt))
            g.append(("AssertZero", nxt + 1))
            nxt += 2
        first_in = n_out
        if kind in ("and", "xor"):
            g.insert(0, ("And" if kind == "and" else "Xor", nxt, first_in, first_in))
        elif kind == "not":
            g.insert(0, ("Not", nxt, first_in))
        elif kind == "copy":
            g.insert(0, ("Copy", nxt, first_in))
        elif kind == "assert_input":
            g.insert(0, ("AssertZero", first_in))
        elif kind == "raw_const":
            g.insert(0, ("Constant", nxt, self.const(ge_p=True)))
        self.funcs.append(ir.Function(name, n_out, n_in, 0, 0, g))
        return (name, n_out, n_in, kind)

    def witnesses(self):
        n = self.n_wit
        self.gates.append(("For", "k", 0, n - 1, [ir.WireRange(0, n - 1)],
                           ("IterExprAnonCall", [("Single", I("k"))], [], 0, 1, [("Witness", 0)])))
        self.next = n
        self.blocks.append((0, n))

    def table_witnesses(self, n):
        """2n wires: the even ones Witness gates, the odd ones irregularly a Witness or an Add.  The even wires' handles are
        an arithmetic progression, their slots are not (input slots are numbered over the inputs only): slot tables"""
        base = self.next
        for k in range(2 * n):
            w = base + k
            if k % 2 == 0 or k < 3 or self.ri(0, 1):
                self.gates.append(("Witness", w))
                self.n_wit += 1
            else:
                self.gates.append(("Add", w, w - 2, w - 1))
        self.next = base + 2 * n
        return base

    def loop(self, f, n_calls=None, carried=False, in_specs=None):
        """in_specs: optional list of (first wire, stride) per input; default: random blocks and strides 0..2"""
        name, n_out, n_in, kind = f
        n = n_calls if n_calls is not None else MIN_CALLS + self.ri(0, 40)
        base = self.next
        S = n_out + self.ri(0, 1)
        if carried:
            self.gates.append(("Add", base, 0, 1))
            base += S
        if n_out > 1 and self.ri(0, 1):
            outs = [("Range", add(C(base), mul(I("i"), C(S))), add(C(base + n_out - 1), mul(C(S), I("i"))))]
        else:
            outs = [("Single", add(C(base + k), mul(I("i"), C(S)))) for k in range(n_out)]
        ins = []
        for k in range(n_in):
            if in_specs is not None:
                first, st = in_specs[k]
            else:
                first, count = self.blocks[self.ri(0, len(self.blocks) - 1)]
                st = self.ri(0, 2)
                while st * (n - 1) >= count:
                    st -= 1
                first += self.ri(0, count - 1 - st * (n - 1))
            if carried and k == 0:
                ins.append(("Single", add(C(base - S), mul(I("i"), C(S)))))
            else:
                ins.append(("Single", add(C(first), mul(I("i"), C(st)))))
        self.gates.append(("For", "i", 0, n - 1, [ir.WireRange(base, base + S * (n - 1) + n_out - 1)],
                           ("IterExprCall", name, outs, ins)))
        self.next = base + S * n
        self.blocks.append((base, S * n) if S == n_out else (base, n_out))
        return base, S

    def tail(self, failing=False):
        for _ in range(4):
            first, count = self.blocks[self.ri(0, len(self.blocks) - 1)]
            t = first + self.ri(0, count - 1)
            s = self.next
            self.gates.append(("MulConstant", s, t, self.le(self.p - 1)))
            self.gates.append(("Add", s + 1, s, t))
            self.gates.append(("AssertZero", s + 1))
            self.next += 2
        if failing:
            first, count = self.blocks[-1]
            self.gates.append(("AssertZero", first + count // 2))   # data dependent, directly on a loop output

    def messages(self, w):
        rel = ir.Relation(self.h, ir.ARITH | ir.BOOL, ir.FOR | ir.FUNCTION | ir.SWITCH, self.funcs, self.gates)
        return [ir.Witness(self.h, [self.le(x) if x < (1 << (8 * self.nb)) else self.le(x % self.p) for x in w]), rel]

    def witness(self):
        if self.raw:   # a quarter of the values >= p (raw integers the reference keeps unreduced)
            return [self.rval(self.p, 1 << (8 * self.nb)) if self.ri(0, 3) == 0 else self.rval(0, self.p) for _ in range(self.n_wit)]
        return [self.rval(0, self.p) for _ in range(self.n_wit)]


def build(p, seed, raw=False, failing=False, n_asserts=None):
    r = ArithRel(p, seed, raw_witness=raw)
    fs = [r.function(f"f{k}", r.ri(1, 3), r.ri(1, 4), "plain", n_asserts if n_asserts is not None else r.ri(0, 2))
          for k in range(r.ri(2, 3))]
    r.witnesses()
    for k in range(r.ri(2, 4)):
        r.loop(fs[r.ri(0, len(fs) - 1)])
    r.tail(failing=failing)
    return r


def record(device, msgs, no_groups=False, **kw):
    z = zkb()
    if no_groups:
        os.environ["ZKB_NO_CALL_GROUPS"] = "1"
    try:
        b = z.GpuBackend(device)
        e = z.Evaluator(b, **kw)
        e.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
    finally:
        os.environ.pop("ZKB_NO_CALL_GROUPS", None)
    return b, e


def handles(e, n):
    out = []
    for w in range(n):
        try:
            out.append(e.value_handle(w))
        except Exception:
            out.append(None)
    return out


def same_state(bg, eg, bs, es, n_wires):
    sg, ss = bg.stats(), bs.stats()
    for k in ("n_asserts", "n_instance", "n_witness", "ir_gates", "callbacks"):
        assert sg[k] == ss[k], k
    assert bg.pending_error() == bs.pending_error()
    hg, hs = handles(eg, n_wires), handles(es, n_wires)
    assert [h is None for h in hg] == [h is None for h in hs]
    for s in range(sg["n_asserts"]):
        assert bg.assert_wire(s) == bs.assert_wire(s), s
    return sg, ss


CASES = [(f, s) for f in FIELDS for s in range(3)]


@pytest.mark.parametrize("field,seed", CASES)
def test_grouped_recording_keeps_the_observable_state(field, seed):
    r = build(FIELDS[field], seed)
    msgs = r.messages(r.witness())
    bg, eg = record(-1, msgs)
    bs, es = record(-1, msgs, no_groups=True)
    sg, ss = same_state(bg, eg, bs, es, r.next)
    assert ss["n_call_groups"] == 0 and sg["n_call_groups"] >= 1
    assert sg["n_values"] < ss["n_values"]
    assert bg.pending_error() is None
    tb = ev.TracingBackend()     # the oracle's trace asks the backend for the same callbacks
    ev.Evaluator.from_messages(msgs, tb)
    oc = tb.counts()
    for k, v in sg["callbacks"].items():
        assert v == oc.get(k, 0), (k, v, oc.get(k, 0))


def test_structural_errors_after_a_group_read_the_same():
    """a gate that rebinds a loop output, and a read of a freed loop output: same pending error text both ways"""
    for tail in ([("Add", 1100, 0, 1)], [("Free", 1100, 1105), ("Add", 10**6, 1101, 1)]):
        r = ArithRel(GOLDILOCKS, 3)
        f = r.function("f", 1, 2, "plain", 1)
        r.witnesses()
        r.loop(f, n_calls=MIN_CALLS, in_specs=[(0, 1), (5, 0)])
        r.gates += tail
        msgs = r.messages(r.witness())
        bg, eg = record(-1, msgs)
        bs, es = record(-1, msgs, no_groups=True)
        assert bg.stats()["n_call_groups"] == 1
        same_state(bg, eg, bs, es, r.next)
        assert bg.pending_error() is not None


def refusal(kind):
    r = ArithRel(BLS12_381_FR, 11)
    n_calls = MIN_CALLS
    f = r.function("f", 2, 2, kind if kind not in ("short", "carried", "switch", "flatten", "expand") else "plain", 1)
    r.witnesses()
    if kind == "short":
        n_calls = MIN_CALLS - 1
    if kind == "switch":     # the loop inside a Switch branch: weighted, refused
        body = [("For", "i", 0, n_calls - 1, [ir.WireRange(2, 2 + 2 * n_calls - 1)],
                 ("IterExprCall", "f", [("Range", add(C(2), mul(I("i"), C(2))), add(C(3), mul(C(2), I("i"))))],
                  [("Single", add(C(1), I("i"))), ("Single", C(1))])),
                ("Add", 0, 2, 3)]
        cond = r.next
        r.gates.append(("Constant", cond, r.le(1)))
        r.gates.append(("Switch", cond, [ir.WireRange(cond + 1, cond + 1)], [r.le(1), r.le(2)],
                        [("AbstractAnonCall", [ir.WireRange(0, n_calls)], 0, 0, body)] * 2))
        r.next = cond + 2
    else:
        r.loop(f, n_calls=n_calls, carried=(kind == "carried"), in_specs=[(0, 1), (3, 0)])
    return r


REFUSALS = ["short", "and", "xor", "not", "copy", "assert_input", "raw_const", "carried", "switch"]


@pytest.mark.parametrize("kind", REFUSALS)
def test_refused_loops_leave_no_group_and_the_same_state(kind):
    r = refusal(kind)
    msgs = r.messages(r.witness())
    bg, eg = record(-1, msgs)
    bs, es = record(-1, msgs, no_groups=True)
    sg, ss = same_state(bg, eg, bs, es, r.next)
    assert sg["n_call_groups"] == 0
    assert sg["n_values"] == ss["n_values"]


@pytest.mark.parametrize("mode", ["flatten", "expand"])
def test_flatten_and_expand_definable_record_no_group(mode):
    r = refusal("plain")
    msgs = r.messages(r.witness())
    kw = {"flatten": True} if mode == "flatten" else {"expand_gate_set": "arithmetic"}
    z = zkb()
    e = z.Evaluator(**kw)
    e.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
    assert e.backend.stats()["n_call_groups"] == 0
    # the same relation evaluated: one group
    bg, _ = record(-1, msgs)
    assert bg.stats()["n_call_groups"] == 1


def test_group_assertions_name_the_local_wire_and_have_no_value():
    r = ArithRel(P127, 4)
    f = r.function("f", 1, 2, "plain", 3)
    body_asserts = [g[1] for g in r.funcs[0].body if g[0] == "AssertZero"]
    r.witnesses()
    s = r.next
    r.gates.append(("MulConstant", s, 0, r.le(0)))
    r.gates.append(("AssertZero", s))                       # seq 0: before the loop
    r.next += 1
    r.loop(f, n_calls=MIN_CALLS + 3, in_specs=[(0, 1), (7, 0)])
    r.gates.append(("AssertZero", s))                       # after the loop
    msgs = r.messages(r.witness())
    b, e = record(-1, msgs)
    st = b.stats()
    assert st["n_call_groups"] == 1
    A = len(body_asserts)
    assert st["n_asserts"] == 2 + (MIN_CALLS + 3) * A
    assert b.assert_wire(0) == s and b.assert_wire(st["n_asserts"] - 1) == s
    for c in (0, 1, MIN_CALLS + 2):
        for k in range(A):
            seq = 1 + c * A + k
            assert b.assert_wire(seq) == body_asserts[k]
            with pytest.raises(zkb().ZkbError, match="call-local wire"):
                b.assert_value(seq)
    assert b.assert_value(0) == b.assert_value(st["n_asserts"] - 1)


def test_plan_hash_does_not_depend_on_plan_threads(monkeypatch):
    r = build(BLS12_381_FR, 7, n_asserts=2)
    msgs = r.messages(r.witness())
    hashes = []
    for t in ("1", "3", "8"):
        monkeypatch.setenv("ZKB_PLAN_THREADS", t)
        b, _ = record(-1, msgs)
        b.finalize(True)
        assert b.stats()["n_call_groups"] >= 1
        hashes.append(b.plan_hash())
    assert len(set(hashes)) == 1


def test_group_registers_are_renamed_by_liveness():
    """a chain of 60 body values, each read once right after it is made: more wires than the device register file holds
    (48), but only a few are live at once, so the loop is still one group"""
    r = ArithRel(GOLDILOCKS, 1)
    g = [("Add", 3, 1, 2)]
    for k in range(60):
        g.append(("MulConstant", 4 + k, 3 + k, r.le(3)))
    g.append(("Add", 0, 63, 1))
    r.funcs.append(ir.Function("chain", 1, 2, 0, 0, g))
    r.witnesses()
    r.loop(("chain", 1, 2, "plain"), n_calls=MIN_CALLS, in_specs=[(0, 1), (2, 0)])
    b, e = record(-1, r.messages(r.witness()))
    b.finalize(True)
    st = b.stats()
    assert st["n_call_groups"] == 1 and st["group_jit_state"] == -1
    assert st["n_values"] < r.n_wit + 2 * MIN_CALLS
