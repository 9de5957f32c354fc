"""Carried loops over prime fields (evaluator.cpp try_call_group, program.h CallGroup::carry): a For loop in which call c
reads output k of call c - d (1 <= d <= kMaxCarryLag = 4), seeded by level-0 values or outputs of earlier groups, is one
call group; so is a loop over an anonymous body of plain gates.  The grouped recording must leave exactly the state the
gate-by-gate unrolling (ZKB_NO_CALL_GROUPS=1) leaves.  Host-only contexts (no GPU)."""
import pytest

from oracle import evaluator as ev
from oracle import fixtures as fx
from oracle import ir
from oracle import sieve_fbs as F
from tests.test_arith_call_groups_host import (BLS12_381_FR, FIELDS, GOLDILOCKS, MIN_CALLS, P127, ArithRel, C, I, add, mul, record,
                                               same_state)
from tests.util import zkb

MAX_LAG = 4
WIDE = {k: v for k, v in FIELDS.items() if v.bit_length() > 64}     # fields of 4 and 8 limbs
NARROW_CHAIN_MIN_CALLS = 1 << 20     # carried loops over 1- and 2-limb fields qualify from here on


class ChainRel(ArithRel):
    """ArithRel with instance values, seed placement and carried loops"""

    def __init__(self, p, seed, n_wit=1100, n_inst=0, raw_witness=False):
        super().__init__(p, seed, n_wit=n_wit, raw_witness=raw_witness)
        self.n_inst = n_inst
        self.group_blocks = []   # (first output wire, S, n_out, n_calls) of the loops recorded as groups
        self.seeded = set()

    def instances(self):
        n = self.n_inst
        base = self.next
        for k in range(n):
            self.gates.append(("Instance", base + k))
        self.next = base + n
        self.blocks.append((base, n))
        return base

    def seed_gate(self, w, source):
        """bind wire w to a level-0 value or an earlier group's output"""
        if source == "witness":
            self.gates.append(("Witness", w))
            self.n_wit += 1
        elif source == "instance":
            self.gates.append(("Copy", w, self.inst0 + self.ri(0, self.n_inst - 1)))
        elif source == "constant":
            self.gates.append(("Constant", w, self.const()))
        elif source == "group":
            first, S, n_out, n = self.group_blocks[self.ri(0, len(self.group_blocks) - 1)]
            self.gates.append(("Copy", w, first + S * self.ri(0, n - 1) + self.ri(0, n_out - 1)))
        elif source == "gate":      # computed by a gate: not ready before the first wavefront, the loop stays unrolled
            self.gates.append(("Add", w, 0, 1))
        else:
            raise ValueError(source)

    def chain(self, f, in_specs, n_calls=None, seeds=None, anon_body=None, S_extra=None):
        """in_specs per input: ("carry", k, lag) | ("aff", first, stride); seeds: the seed source per carried input.
        anon_body: the loop's body as an IterExprAnonCall of these gates instead of a call of f"""
        name, n_out, n_in, _ = f
        n = n_calls if n_calls is not None else MIN_CALLS + self.ri(0, 40)
        S = n_out + (S_extra if S_extra is not None else self.ri(0, 1))
        lags = [s[2] for s in in_specs if s[0] == "carry"]
        back = max([l for l in lags if l > 0] + [0])
        base = self.next + S * back
        j = 0
        for s in in_specs:
            if s[0] != "carry":
                continue
            _, k, lag = s
            src = seeds[j] if seeds else ["witness", "instance", "constant", "group"][self.ri(0, 3 if self.group_blocks else 2)]
            if src == "instance" and not self.n_inst:
                src = "witness"
            for c in range(max(lag, 0)):
                w = base + k - S * lag + S * c
                if w < base and w not in self.seeded:   # two inputs carrying one output share seeds
                    self.seed_gate(w, src)
                    self.seeded.add(w)
            j += 1
        outs = [("Single", add(C(base + k), mul(I("i"), C(S)))) for k in range(n_out)]
        ins = []
        for s in in_specs:
            if s[0] == "carry":
                _, k, lag = s
                ins.append(("Single", add(C(base + k - S * lag), mul(I("i"), C(S)))))
            else:
                _, first, st = s
                ins.append(("Single", add(C(first), mul(I("i"), C(st)))))
        body = ("IterExprCall", name, outs, ins) if anon_body is None else ("IterExprAnonCall", outs, ins, 0, 0, anon_body)
        self.gates.append(("For", "i", 0, n - 1, [ir.WireRange(base, base + S * (n - 1) + n_out - 1)], body))
        self.next = base + S * n
        self.blocks.append((base, S * n) if S == n_out else (base, n_out))
        self.group_blocks.append((base, S, n_out, n))
        return base, S

    def messages(self, w, inst=None):
        m = super().messages(w)
        if self.n_inst:
            vals = inst if inst is not None else self.instance_values()
            m.insert(0, ir.Instance(self.h, [self.le(x) for x in vals]))
        return m

    def instance_values(self):
        return [self.rval(0, self.p) for _ in range(self.n_inst)]


def random_specs(r, n_out, n_in, n):
    """at least one carried input; the rest affine (strides 0..2) over the witness block"""
    specs = []
    for k in range(n_in):
        if k == 0 or r.ri(0, 1):
            specs.append(("carry", r.ri(0, n_out - 1), r.ri(1, MAX_LAG)))
        else:
            first, count = r.blocks[0]
            st = r.ri(0, 2)
            while st * (n - 1) >= count:
                st -= 1
            specs.append(("aff", first + r.ri(0, count - 1 - st * (n - 1)), st))
    return specs


def anon_body_of(r, f):
    return next(fn for fn in r.funcs if fn.name == f[0]).body


def build_chains(p, seed, n_asserts=None, raw=False, failing=False):
    """a plain group, then carried loops (named and anonymous) seeded from witnesses, instances, constants and that
    group's outputs; a tail that reads the chains' outputs"""
    r = ChainRel(p, seed, n_inst=8, raw_witness=raw)
    fs = [r.function(f"f{k}", r.ri(1, 3), r.ri(1, 4), "plain", n_asserts if n_asserts is not None else r.ri(0, 2)) for k in range(3)]
    r.witnesses()
    r.inst0 = r.instances()
    g = fs[0]
    base, S = r.loop(g, n_calls=MIN_CALLS, in_specs=[(0, 1)] * g[2])
    r.group_blocks.append((base, S, g[1], MIN_CALLS))
    n_chains = r.ri(2, 3)
    for c in range(n_chains):
        f = fs[1 + c % 2]
        n = MIN_CALLS + r.ri(0, 40)
        specs = random_specs(r, f[1], f[2], n)
        r.chain(f, specs, n_calls=n, anon_body=anon_body_of(r, f) if c % 2 else None)
    r.tail(failing=failing)
    return r, n_chains


def compare(r, inst=None):
    msgs = r.messages(r.witness(), inst)
    bg, eg = record(-1, msgs)
    bs, es = record(-1, msgs, no_groups=True)
    sg, ss = same_state(bg, eg, bs, es, r.next)
    assert ss["n_call_groups"] == 0 and ss["n_carried_groups"] == 0
    return msgs, bg, sg, ss


CASES = [(f, s) for f in FIELDS for s in range(3)]


@pytest.mark.parametrize("field,seed", CASES)
def test_carried_recording_keeps_the_observable_state(field, seed):
    """over 1- and 2-limb fields these chains are shorter than the minimum: they stay unrolled, the plain group remains"""
    r, n_chains = build_chains(FIELDS[field], seed)
    msgs, bg, sg, ss = compare(r)
    if field not in WIDE:
        n_chains = 0
    assert sg["n_carried_groups"] == n_chains and sg["n_call_groups"] == 1 + n_chains
    assert sg["n_values"] < ss["n_values"]
    assert bg.pending_error() is None
    tb = ev.TracingBackend()
    ev.Evaluator.from_messages(msgs, tb)
    oc = tb.counts()
    for k, v in sg["callbacks"].items():
        assert v == oc.get(k, 0), (k, v, oc.get(k, 0))
    bg.finalize(True)
    st = bg.stats()
    assert st["n_carried_groups"] == n_chains and st["n_group_launches"] >= 1 + (n_chains > 0)


@pytest.mark.parametrize("lag", range(1, MAX_LAG + 1))
@pytest.mark.parametrize("source", ["witness", "instance", "constant", "group"])
def test_every_lag_and_seed_source(lag, source):
    r = ChainRel(P127, 10 * lag, n_inst=4)
    f = r.function("h", 2, 3, "plain", 1)
    r.witnesses()
    r.inst0 = r.instances()
    if source == "group":
        base, S = r.loop(f, n_calls=MIN_CALLS, in_specs=[(0, 1), (1, 1), (5, 0)])
        r.group_blocks.append((base, S, 2, MIN_CALLS))
    r.chain(f, [("carry", 1, lag), ("aff", 3, 0), ("carry", 0, 1 + lag % MAX_LAG)], n_calls=MIN_CALLS + lag,
            seeds=[source, source])
    _, bg, sg, _ = compare(r)
    assert sg["n_carried_groups"] == 1 and sg["n_call_groups"] == 1 + (source == "group")


def test_anonymous_non_carried_loop_is_a_group():
    r = ChainRel(P127, 5)
    f = r.function("f", 1, 2, "plain", 2)
    r.witnesses()
    r.chain(f, [("aff", 0, 1), ("aff", 9, 0)], n_calls=MIN_CALLS, anon_body=anon_body_of(r, f))
    _, _, sg, _ = compare(r)
    assert sg["n_call_groups"] == 1 and sg["n_carried_groups"] == 0


def test_anonymous_bodies_that_consume_values_or_nest_are_refused():
    r = ChainRel(GOLDILOCKS, 6)
    f = r.function("f", 1, 2, "plain", 0)
    r.witnesses()
    n_wit0 = r.n_wit
    body = [("Witness", 40), ("Add", 41, 40, 1)] + anon_body_of(r, f)
    base = r.next
    n = MIN_CALLS
    outs = [("Single", add(C(base), I("i")))]
    ins = [("Single", add(C(0), I("i"))), ("Single", C(3))]
    r.gates.append(("For", "i", 0, n - 1, [ir.WireRange(base, base + n - 1)], ("IterExprAnonCall", outs, ins, 0, 1, body)))
    r.next = base + n
    r.n_wit = n_wit0 + n
    _, _, sg, ss = compare(r)
    assert sg["n_call_groups"] == 0 and sg["n_values"] == ss["n_values"]


def refusal(kind):
    r = ChainRel(BLS12_381_FR, 11)
    f = r.function("f", 2, 2, "plain", 1)
    r.witnesses()
    n = MIN_CALLS - 1 if kind == "short" else MIN_CALLS
    if kind == "gate_seed":
        r.chain(f, [("carry", 0, 2), ("aff", 3, 0)], n_calls=n, seeds=["gate"])
    elif kind == "lag0":            # reads its own call's output: unbound when the call starts
        r.chain(f, [("carry", 0, 0), ("aff", 3, 0)], n_calls=n)
    elif kind == "lag5":
        r.chain(f, [("carry", 1, MAX_LAG + 1), ("aff", 3, 0)], n_calls=n, seeds=["witness"])
    elif kind == "later":           # call c reads output 0 of call c + 1
        r.chain(f, [("carry", 0, -1), ("aff", 3, 0)], n_calls=n)
    elif kind == "stride":          # input stride 2S: partly seeds, partly outputs of no fixed lag
        base, S = r.next + 4, 2
        for w in range(r.next, base):
            r.gates.append(("Witness", w))
            r.n_wit += 1
        outs = [("Single", add(C(base + k), mul(I("i"), C(S)))) for k in range(2)]
        ins = [("Single", add(C(base - 2), mul(I("i"), C(2 * S)))), ("Single", C(3))]
        r.gates.append(("For", "i", 0, n - 1, [ir.WireRange(base, base + S * n - 1)], ("IterExprCall", "f", outs, ins)))
        r.next = base + S * n
    elif kind == "short":
        r.chain(f, [("carry", 0, 1), ("aff", 3, 0)], n_calls=n, seeds=["witness"])
    elif kind == "switch":          # a carried loop inside a Switch branch (seeded by the branch's input 2): weighted, refused
        body = [("For", "i", 0, n - 1, [ir.WireRange(4, 4 + 2 * n - 1)],
                 ("IterExprCall", "f", [("Range", add(C(4), mul(I("i"), C(2))), add(C(5), mul(C(2), I("i"))))],
                  [("Single", add(C(2), mul(I("i"), C(2)))), ("Single", C(1))])),
                ("Add", 0, 4, 5)]
        cond = r.next
        r.gates.append(("Constant", cond, r.le(1)))
        r.gates.append(("Switch", cond, [ir.WireRange(cond + 1, cond + 1)], [r.le(1), r.le(2)],
                        [("AbstractAnonCall", [ir.WireRange(0, 1)], 0, 0, body)] * 2))
        r.next = cond + 2
    return r


REFUSALS = ["gate_seed", "lag0", "lag5", "later", "stride", "short", "switch"]


@pytest.mark.parametrize("kind", REFUSALS)
def test_refused_carried_loops_leave_no_group_and_the_same_state(kind):
    r = refusal(kind)
    msgs, bg, sg, ss = compare(r)
    assert sg["n_call_groups"] == 0 and sg["n_carried_groups"] == 0
    assert sg["n_values"] == ss["n_values"]
    if kind in ("lag0", "later"):
        assert bg.pending_error() is not None and "No value given" in bg.pending_error()


@pytest.mark.parametrize("mode", ["flatten", "expand"])
def test_flatten_and_expand_definable_record_no_carried_group(mode):
    r = ChainRel(BLS12_381_FR, 11)
    f = r.function("f", 2, 2, "plain", 1)
    r.witnesses()
    r.chain(f, [("carry", 0, 1), ("aff", 3, 0)], n_calls=MIN_CALLS, seeds=["witness"])
    msgs = r.messages(r.witness())
    kw = {"flatten": True} if mode == "flatten" else {"expand_gate_set": "arithmetic"}
    z = zkb()
    e = z.Evaluator(**kw)
    e.ingest_source(z.Source.from_buffers([F.write_messages(msgs)]))
    assert e.backend.stats()["n_call_groups"] == 0
    bg, _ = record(-1, msgs)
    assert bg.stats()["n_carried_groups"] == 1


@pytest.mark.parametrize("n_calls", [MIN_CALLS, NARROW_CHAIN_MIN_CALLS - 1, NARROW_CHAIN_MIN_CALLS])
def test_narrow_field_chains_need_more_calls(n_calls):
    r = ChainRel(GOLDILOCKS, 8)
    f = ("h", 1, 2, "plain")
    r.funcs.append(ir.Function("h", 1, 2, 0, 0, [("Mul", 3, 1, 2), ("AddConstant", 0, 3, r.le(1))]))
    r.witnesses()
    r.chain(f, [("carry", 0, 1), ("aff", 0, 0)], n_calls=n_calls, seeds=["witness"], S_extra=0)
    msgs = r.messages(r.witness())
    b, _ = record(-1, msgs)
    assert b.stats()["n_carried_groups"] == (n_calls >= NARROW_CHAIN_MIN_CALLS)
    if n_calls == MIN_CALLS:
        compare(r)


def test_carried_loop_over_p2_stays_unrolled():
    r = ChainRel(2, 12)
    r.funcs.append(ir.Function("x", 1, 2, 0, 0, [("Xor", 0, 1, 2)]))
    r.witnesses()
    r.chain(("x", 1, 2, "plain"), [("carry", 0, 1), ("aff", 0, 1)], n_calls=MIN_CALLS, seeds=["witness"])
    _, _, sg, ss = compare(r)
    assert sg["n_call_groups"] == 0 and sg["n_values"] == ss["n_values"]


def test_reference_example_records_as_before():
    """its loops (Fibonacci over an anonymous body, com.example::mul over i-1, i-2) are seeded by computed wires and are
    shorter than the minimum: gate by gate, as before"""
    msgs = [fx.example_instance(), fx.example_witness(), fx.example_relation()]
    bg, eg = record(-1, msgs)
    bs, es = record(-1, msgs, no_groups=True)
    sg, _ = same_state(bg, eg, bs, es, 64)
    assert sg["n_call_groups"] == 0 and sg["n_carried_groups"] == 0
    assert bg.stats()["n_values"] == bs.stats()["n_values"]


def chain_then_group(p, seed=21):
    """depth 0: a plain group; depth 1: a chain seeded by its outputs; depth 2: a plain group that reads the chain's outputs
    (stride S over the chain's block); a tail that reads all three"""
    r = ChainRel(p, seed)
    g0 = r.function("g0", 1, 2, "plain", 1)
    f = r.function("f", 2, 2, "plain", 1)
    g1 = r.function("g1", 1, 2, "plain", 1)
    r.witnesses()
    base, S = r.loop(g0, n_calls=MIN_CALLS, in_specs=[(0, 1), (1, 1)])
    r.group_blocks.append((base, S, 1, MIN_CALLS))
    cb, cs = r.chain(f, [("carry", 1, 2), ("aff", 5, 1)], n_calls=MIN_CALLS + 7, seeds=["group"])
    r.loop(g1, n_calls=MIN_CALLS, in_specs=[(cb, cs), (cb + 1, cs)])
    r.tail()
    return r


def test_a_group_reading_a_chain_runs_after_it():
    r = chain_then_group(P127)
    msgs, bg, sg, _ = compare(r)
    assert sg["n_call_groups"] == 3 and sg["n_carried_groups"] == 1
    bg.finalize(True)
    assert bg.stats()["n_group_launches"] == 3       # one launch per depth: group, chain, group


def plan_hash(msgs):
    b, _ = record(-1, msgs)
    b.finalize(True)
    assert b.stats()["n_carried_groups"] == 1
    return b.plan_hash()


def test_plan_hash_tells_lags_and_seeds_apart():
    hashes = []
    for lag, src in ((1, "witness"), (2, "witness"), (1, "constant")):
        r = ChainRel(P127, 5)
        f = r.function("f", 1, 2, "plain", 0)
        r.witnesses()
        r.chain(f, [("carry", 0, lag), ("aff", 0, 1)], n_calls=MIN_CALLS, seeds=[src], S_extra=0)
        hashes.append(plan_hash(r.messages(r.witness())))
    assert len(set(hashes)) == 3


def test_plan_hash_covers_the_chains(monkeypatch):
    r, _ = build_chains(BLS12_381_FR, 7, n_asserts=2)
    msgs = r.messages(r.witness())
    hashes = []
    for t in ("1", "3"):
        monkeypatch.setenv("ZKB_PLAN_THREADS", t)
        b, _ = record(-1, msgs)
        b.finalize(True)
        hashes.append(b.plan_hash())
    assert len(set(hashes)) == 1
