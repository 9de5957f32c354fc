"""Synthetic workloads of BASELINE.json's configs (numpy, deterministic).

These are the INPUTS of the benchmark and of the parity tests — flat relations in the
`zkb_gate` array form (the simple arms of the reference's `Gate`,
rust/src/structs/gates.rs:18-45) plus witness vectors.  Nothing here evaluates a gate.

random_circuit  "random Add/Mul/AssertZero circuit" (configs C2, C3), SURVEY.md section 8(d):
    wires 0..n_in-1   Witness: x_0 .. x_{h-1}, then x'_0 .. x'_{h-1} with x'_i = p - x_i   (not counted gates)
    then slots drawn 41 % Add, 41 % Mul, 18 % assertion; operands uniform over all earlier wires (or over the last
    `window` of them).  Every wire w has a twin w' whose value is sign(w) * value(w), sign in {+1, -1}:
      Add / Mul slot  g = op(a, b) and its twin g' = op(a', b')          (2 counted gates; Add needs sign(a) = sign(b),
                      so b is snapped to the nearest earlier wire with a's sign; sign(Mul) = sign(a) * sign(b))
      assertion slot  s = Add(t, t'); AssertZero(s) on an arbitrary earlier wire t with sign -1   (2 counted gates)
    so an assertion holds iff the witness is consistent (x'_i = -x_i) AND every gate in the cones of t and t' was
    computed correctly: a wrong value anywhere upstream makes t + t' non-zero.  This is section 8(d)'s
    witness-dependent assertion `Witness(k) = p - v(t); s = Add(t, k); AssertZero(s)` with k computed inside the circuit
    by the twin gates instead of being shipped as one extra witness value per assertion: at C3's size that would be
    1.5 M x 32 B = 48 MB per witness, 196 GB for the batch of 4096 -- more than a B200's HBM, let alone beside the
    wire store.  A gate and its twin share no operand, but operands are drawn independently, so the readers of one wire
    do coincide: at 2^24, 37 % of the operand reads inside a wavefront repeat a wire another gate of that wavefront reads
    (scripts/wavefront_reuse_model.py).  There are no constants.  Gate histogram:
    Add 50 %, Mul 41 %, AssertZero 9 % of `n_gates` (section 8(d)'s mix).
    Corrupting the mirror x'_k of a tracked input (k < n_tracked <= 64) makes every assertion whose t depends on x_k or
    x'_k fail (up to a 2^-250 coincidence): the first such assertion in program order is known from a taint pass
    done while generating (`first_fail_of_input`), and the tests confirm it with the oracle.
    Generated block-wise with numpy: the operands of a block come from earlier blocks only (blocks of 1/8 of the
    wires that exist, at most 4096 slots), which is what lets the signs and taints be propagated vectorised.
"""
from __future__ import annotations

import numpy as np

GATE_DTYPE = np.dtype([("op", "u1"), ("pad", "u1", (3,)), ("out", "<u4"), ("a", "<u4"), ("b", "<u4")])
(G_CONSTANT, G_ASSERT_ZERO, G_COPY, G_ADD, G_MUL, G_ADD_CONSTANT, G_MUL_CONSTANT, G_AND, G_XOR, G_NOT, G_INSTANCE,
 G_WITNESS, G_FREE) = range(1, 14)

GOLDILOCKS = (1 << 64) - (1 << 32) + 1
BLS12_381_FR = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
BN254_FR = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001


def elem_bytes(p: int) -> int:
    bits = p.bit_length()
    return 4 if bits <= 32 else 8 if bits <= 64 else 16 if bits <= 128 else 32


def le_bytes(v: int, n: int) -> np.ndarray:
    return np.frombuffer(int(v).to_bytes(n, "little"), dtype=np.uint8)


class FlatCircuit:
    def __init__(self):
        self.p = 0
        self.gates = None          # GATE_DTYPE
        self.const_pool = None     # uint8 [n_consts, stride] (empty: the circuit has no constants)
        self.n_inputs = 0          # Witness gates: x_0 .. x_{h-1}, then their mirrors x'_i = -x_i
        self.n_gates = 0           # counted gates: Add + Mul + AssertZero
        self.n_wires = 0
        self.n_tracked = 0         # inputs 0 .. n_tracked-1 can be corrupted with a known first failing assertion
        self.first_fail_of_input = None  # assert seq of the first assertion that sees tracked input k (-1: none)
        self.n_asserts = 0
        self.hist = {}


def _block_size(pool: int, window: int) -> int:
    span = min(pool, window) if window else pool
    return int(min(4096, max(4, span // 8)))


def random_circuit(n_gates: int, n_inputs: int, p: int, seed: int, n_tracked: int = 32, window: int = 0,
                   assert_frac: float = 0.18) -> FlatCircuit:
    """See the module docstring.  n_gates must be even (every slot costs two counted gates)."""
    if n_gates % 2 or n_gates < 2:
        raise ValueError("n_gates must be even")
    if n_inputs < 2:
        raise ValueError("at least two inputs (one value and its mirror)")
    rng = np.random.default_rng(seed)
    h = n_inputs // 2
    n_in = 2 * h
    n_slots = n_gates // 2
    n_tracked = min(n_tracked, h, 64)
    kinds_all = rng.choice(3, size=n_slots, p=[(1 - assert_frac) / 2, (1 - assert_frac) / 2, assert_frac]).astype(np.int8)
    n_emit = n_in + n_gates
    g = np.zeros(n_emit, dtype=GATE_DTYPE)
    g["op"][:n_in] = G_WITNESS
    g["out"][:n_in] = np.arange(n_in, dtype=np.uint32)
    # the pool: every wire an operand may be drawn from, with the wire that holds its negated-or-equal twin
    cap = n_in + 2 * n_slots
    pool_wire = np.empty(cap, dtype=np.int64)
    pool_partner = np.empty(cap, dtype=np.int64)
    pool_sign = np.empty(cap, dtype=np.int8)        # value(partner) = sign * value(wire)
    pool_taint = np.zeros(cap, dtype=np.uint64)      # which tracked inputs (either twin) the wire depends on
    last_minus = np.empty(cap, dtype=np.int64)       # largest pool index <= i with sign -1 / +1 (-1: none)
    last_plus = np.empty(cap, dtype=np.int64)
    pool_wire[:n_in] = np.arange(n_in)
    pool_partner[:h] = np.arange(h, n_in)
    pool_partner[h:n_in] = np.arange(h)
    pool_sign[:n_in] = -1
    bits = np.uint64(1) << np.arange(n_tracked, dtype=np.uint64)
    pool_taint[:n_tracked] = bits
    pool_taint[h:h + n_tracked] = bits
    last_minus[:n_in] = np.arange(n_in)
    last_plus[:n_in] = -1
    P = n_in                 # pool size
    n_wires = n_in
    e = n_in                 # gates emitted
    n_asserts = 0
    first_fail = np.full(n_tracked, -1, dtype=np.int64)
    missing = np.uint64((1 << n_tracked) - 1) if n_tracked else np.uint64(0)
    s0 = 0
    while s0 < n_slots:
        B = min(_block_size(P, window), n_slots - s0)
        k = kinds_all[s0:s0 + B].copy()
        lo = max(0, P - window) if window else 0
        ia = lo + (rng.random(B) * (P - lo)).astype(np.int64)
        ib = lo + (rng.random(B) * (P - lo)).astype(np.int64)
        sa = pool_sign[ia]
        # Add needs operands of equal sign: snap b down to the nearest wire with a's sign (never a's own twin, whose
        # sum with a would be the constant zero); where there is none the slot becomes a Mul
        is_add = k == 0
        snapped = np.where(sa < 0, last_minus[ib], last_plus[ib])
        twin = is_add & (snapped == pool_partner[ia])
        below = np.maximum(snapped - 1, 0)
        snapped = np.where(twin, np.where(snapped > 0, np.where(sa < 0, last_minus[below], last_plus[below]), -1), snapped)
        to_mul = is_add & ((snapped < 0) | (snapped == pool_partner[ia]))
        k[to_mul] = 1
        is_add = k == 0
        ib = np.where(is_add, snapped, ib)
        # assertion slots test a wire t whose twin holds -t
        is_as = k == 2
        it = last_minus[ia]
        am = ~is_as
        n_am = int(am.sum())
        n_as = B - n_am
        j = np.arange(B)
        rank_am = np.cumsum(am) - 1
        cost1 = np.where(is_as, 2, 1)
        off1 = e + np.cumsum(cost1) - cost1
        wire1 = n_wires + j
        # ---- phase 1: the gates of the block in slot order
        sel = np.flatnonzero(am)
        gi = off1[sel]
        a_idx, b_idx = ia[sel], ib[sel]
        g["op"][gi] = np.where(k[sel] == 0, G_ADD, G_MUL)
        g["out"][gi] = wire1[sel]
        g["a"][gi] = pool_wire[a_idx]
        g["b"][gi] = pool_wire[b_idx]
        asel = np.flatnonzero(is_as)
        if n_as:
            gi = off1[asel]
            t = it[asel]
            g["op"][gi] = G_ADD
            g["out"][gi] = wire1[asel]
            g["a"][gi] = pool_wire[t]
            g["b"][gi] = pool_wire[pool_partner[t]]
            g["op"][gi + 1] = G_ASSERT_ZERO
            g["a"][gi + 1] = wire1[asel]
            if missing:
                tm = pool_taint[t]
                if np.bitwise_or.reduce(tm) & missing:
                    for q in range(n_as):
                        hit = tm[q] & missing
                        if hit:
                            for bit in range(n_tracked):
                                if (int(hit) >> bit) & 1:
                                    first_fail[bit] = n_asserts + q
                            missing = missing & ~hit
            n_asserts += n_as
        # ---- phase 2: the twins of the block's Add / Mul gates, on the twins of their operands
        e2 = e + int(cost1.sum())
        gi = e2 + np.arange(n_am)
        wire2 = n_wires + B + np.arange(n_am)
        g["op"][gi] = g["op"][off1[sel]]
        g["out"][gi] = wire2
        g["a"][gi] = pool_wire[pool_partner[a_idx]]
        g["b"][gi] = pool_wire[pool_partner[b_idx]]
        # ---- the block's wires join the pool
        sgn = np.where(k[sel] == 0, sa[sel], sa[sel] * pool_sign[b_idx]).astype(np.int8)
        tnt = pool_taint[a_idx] | pool_taint[b_idx]
        lo_p, mid_p, hi_p = P, P + n_am, P + 2 * n_am
        pool_wire[lo_p:mid_p] = wire1[sel]
        pool_wire[mid_p:hi_p] = wire2
        pool_partner[lo_p:mid_p] = np.arange(mid_p, hi_p)
        pool_partner[mid_p:hi_p] = np.arange(lo_p, mid_p)
        pool_sign[lo_p:mid_p] = sgn
        pool_sign[mid_p:hi_p] = sgn
        pool_taint[lo_p:mid_p] = tnt
        pool_taint[mid_p:hi_p] = tnt
        idx = np.arange(lo_p, hi_p)
        s2 = pool_sign[lo_p:hi_p]
        last_minus[lo_p:hi_p] = np.maximum(np.maximum.accumulate(np.where(s2 < 0, idx, -1)), last_minus[lo_p - 1])
        last_plus[lo_p:hi_p] = np.maximum(np.maximum.accumulate(np.where(s2 > 0, idx, -1)), last_plus[lo_p - 1])
        P = hi_p
        n_wires += B + n_am
        e = e2 + n_am
        s0 += B
    assert e == n_emit, (e, n_emit)
    if n_wires >= (1 << 32) - 16:
        raise ValueError("circuit too large for 32-bit wire ids")

    c = FlatCircuit()
    c.p = p
    c.gates = g
    c.const_pool = np.zeros((0, elem_bytes(p)), dtype=np.uint8)
    c.n_inputs = n_in
    c.n_gates = n_gates
    c.n_wires = n_wires
    c.n_tracked = n_tracked
    c.first_fail_of_input = first_fail
    c.n_asserts = n_asserts
    c.hist = {"add": int((g["op"] == G_ADD).sum()), "mul": int((g["op"] == G_MUL).sum()), "assert_zero": n_asserts}
    assert c.hist["add"] + c.hist["mul"] + n_asserts == n_gates
    return c


def _limbs_of(p: int, nl: int) -> np.ndarray:
    return np.array([(p >> (32 * i)) & 0xFFFFFFFF for i in range(nl)], dtype=np.uint64)


def random_field_elements(rng, shape, p: int) -> np.ndarray:
    """uniform in [0, p) by rejection; returns uint8 [*shape, elem_bytes(p)] little-endian"""
    eb = elem_bytes(p)
    n = int(np.prod(shape))
    bits = p.bit_length()
    nl = eb // 4
    plimbs = _limbs_of(p, nl).astype(np.uint32)
    out = np.zeros((n, nl), dtype=np.uint32)
    todo = np.arange(n)
    top_bits = bits - 32 * (nl - 1)
    top_mask = np.uint32((1 << top_bits) - 1) if top_bits < 32 else np.uint32(0xFFFFFFFF)
    while len(todo):
        cand = rng.integers(0, 1 << 32, size=(len(todo), nl), dtype=np.uint64).astype(np.uint32)
        cand[:, nl - 1] &= top_mask
        # cand < p, lexicographic from the top limb
        lt = np.zeros(len(todo), dtype=bool)
        eq = np.ones(len(todo), dtype=bool)
        for i in range(nl - 1, -1, -1):
            lt |= eq & (cand[:, i] < plimbs[i])
            eq &= cand[:, i] == plimbs[i]
        out[todo[lt]] = cand[lt]
        todo = todo[~lt]
    return out.view(np.uint8).reshape(*shape, eb)


def negate_mod(x: np.ndarray, p: int) -> np.ndarray:
    """(p - x) mod p limb-wise for uint8 [..., elem_bytes(p)] little-endian values below p"""
    eb = x.shape[-1]
    nl = eb // 4
    xl = np.ascontiguousarray(x).view(np.uint32).reshape(-1, nl).astype(np.uint64)
    pl = _limbs_of(p, nl)
    out = np.zeros_like(xl)
    borrow = np.zeros(len(xl), dtype=np.uint64)
    for i in range(nl):
        d = pl[i] + (np.uint64(1) << np.uint64(32)) - xl[:, i] - borrow
        out[:, i] = d & np.uint64(0xFFFFFFFF)
        borrow = np.uint64(1) - (d >> np.uint64(32))
    out[(xl == 0).all(axis=1)] = 0
    return out.astype(np.uint32).view(np.uint8).reshape(x.shape)


def make_witnesses(c: FlatCircuit, n_batch: int, seed: int, corrupt=None) -> np.ndarray:
    """uint8 [n_batch, n_inputs, elem_bytes]: x_0 .. x_{h-1} uniform, then the mirrors x'_i = p - x_i.
    corrupt: {witness index: tracked input k} -> x'_k is off by one for that witness."""
    rng = np.random.default_rng(seed ^ 0x5EED)
    eb = elem_bytes(c.p)
    h = c.n_inputs // 2
    w = np.empty((n_batch, c.n_inputs, eb), dtype=np.uint8)
    w[:, :h, :] = random_field_elements(rng, (n_batch, h), c.p)
    w[:, h:, :] = negate_mod(w[:, :h, :], c.p)
    for j, k in (corrupt or {}).items():
        if k >= c.n_tracked:
            raise ValueError("only the tracked inputs can be corrupted")
        y = (int.from_bytes(w[j, h + k].tobytes(), "little") + 1) % c.p
        w[j, h + k, :] = le_bytes(y, eb)
    return w


def expected_first_fail(c: FlatCircuit, n_batch: int, corrupt=None) -> np.ndarray:
    """first failing assert seq per witness (-1: TRUE): the first assertion, in program order, on a wire that
    depends on the corrupted input or on its twin"""
    out = np.full(n_batch, -1, dtype=np.int64)
    for j, k in (corrupt or {}).items():
        out[j] = int(c.first_fail_of_input[k])
    return out


def algorithmic_bytes_per_witness(c: FlatCircuit) -> int:
    """SURVEY.md section 8(d): Add/Mul = 3E, AssertZero = E"""
    E = elem_bytes(c.p)
    return 3 * E * (c.hist["add"] + c.hist["mul"]) + E * c.hist["assert_zero"]


# ---------------------------------------------------------------------------------------------
# C4: "multiplication-gate" shaped R1CS (SURVEY.md section 8d)
# ---------------------------------------------------------------------------------------------
class R1cs:
    def __init__(self):
        self.p = 0
        self.n_rows = 0
        self.n_vars = 0
        self.n_free = 0
        self.A = self.B = self.C = None   # (row_ptr uint64, col uint32, coef_idx uint32)
        self.coef_table = None            # uint8 [n_coefs, elem_bytes]
        self.coefs = None                 # python ints
        self.nnz = 0


def random_r1cs(n_rows: int, n_free: int, p: int, seed: int) -> R1cs:
    """Row r: (A_r . z)(B_r . z) = z[s_r] with s_r = n_free + 1 + r a fresh slack variable.
    A_r, B_r: 1 + Poisson(2) terms (capped at 8) over uniformly chosen ids < s_r; coefficients from a
    seeded 256-entry table plus {1, p-1}.  Variable 0 is the constant one."""
    rng = np.random.default_rng(seed)
    eb = elem_bytes(p)
    coefs = [1, p - 1] + [int.from_bytes(rng.bytes(eb), "little") % p for _ in range(256)]
    r = R1cs()
    r.p = p
    r.n_rows = n_rows
    r.n_free = n_free
    r.n_vars = 1 + n_free + n_rows
    r.coefs = coefs
    r.coef_table = np.stack([le_bytes(c, eb) for c in coefs])
    mats = []
    for _ in range(2):
        cnt = np.minimum(1 + rng.poisson(2.0, size=n_rows), 8).astype(np.int64)
        row_ptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint64)
        nnz = int(row_ptr[-1])
        rows = np.repeat(np.arange(n_rows, dtype=np.int64), cnt)
        limit = n_free + 1 + rows                       # ids < s_r
        col = (rng.random(nnz) * limit).astype(np.int64).astype(np.uint32)
        ci = rng.integers(0, len(coefs), size=nnz).astype(np.uint32)
        # half of the coefficients are the literal 1, as in real R1CS
        ci[rng.random(nnz) < 0.5] = 0
        mats.append((row_ptr, col, ci))
    r.A, r.B = mats
    r.C = (np.arange(n_rows + 1, dtype=np.uint64), (n_free + 1 + np.arange(n_rows)).astype(np.uint32),
           np.zeros(n_rows, dtype=np.uint32))
    r.nnz = int(r.A[0][-1] + r.B[0][-1] + n_rows)
    return r


def r1cs_assignment(r: R1cs, seed: int):
    """A satisfying assignment z (python ints): free variables random, slack z[s_r] := (A_r.z)(B_r.z) mod p."""
    rng = np.random.default_rng(seed ^ 0xA551)
    p = r.p
    free = random_field_elements(rng, (r.n_free,), p)
    z = [1] + [int.from_bytes(free[i].tobytes(), "little") for i in range(r.n_free)] + [0] * r.n_rows
    coefs = r.coefs
    (rpa, ca, ia), (rpb, cb, ib) = r.A, r.B
    rpa, ca, ia, rpb, cb, ib = (x.tolist() for x in (rpa, ca, ia, rpb, cb, ib))
    base = r.n_free + 1
    for row in range(r.n_rows):
        a = 0
        for e in range(rpa[row], rpa[row + 1]):
            a += coefs[ia[e]] * z[ca[e]]
        b = 0
        for e in range(rpb[row], rpb[row + 1]):
            b += coefs[ib[e]] * z[cb[e]]
        z[base + row] = (a % p) * (b % p) % p
    return z


def assignment_bytes(z, p: int) -> np.ndarray:
    eb = elem_bytes(p)
    buf = b"".join(int(v).to_bytes(eb, "little") for v in z)
    return np.frombuffer(buf, dtype=np.uint8).reshape(len(z), eb).copy()


def r1cs_first_row_reading(r: R1cs, var: int) -> int:
    """first row whose A, B or C mentions variable `var`"""
    best = r.n_rows
    for rp, col, _ in (r.A, r.B, r.C):
        hits = np.flatnonzero(col == var)
        if len(hits):
            row = int(np.searchsorted(rp, hits[0], side="right") - 1)
            best = min(best, row)
    return best


def r1cs_algorithmic_bytes(r: R1cs) -> int:
    """SURVEY.md section 8(d): per nnz 4 B col + 4 B coef index + E gathered z; per row 3 x 4 B row_ptr"""
    return (8 + elem_bytes(r.p)) * r.nnz + 12 * r.n_rows


def r1cs_gate_equivalent(r: R1cs) -> int:
    """gates `zkif-to-ir` emits for this system: 2 per term with id != 0 (Constant + Mul), 1 per id-0 term,
    (terms - 1) Adds per LC, 4 per row (from_r1cs.rs:71-125)"""
    total = 0
    for rp, col, _ in (r.A, r.B, r.C):
        total += int(2 * (col != 0).sum() + (col == 0).sum())
        cnt = np.diff(rp.astype(np.int64))
        total += int(np.maximum(cnt - 1, 0).sum() + (cnt == 0).sum())
    return total + 4 * r.n_rows
