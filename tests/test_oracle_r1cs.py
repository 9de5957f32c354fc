"""Pins oracle/r1cs.py, the direct statement of the R1CS check that tests/test_gpu_r1cs_reference.py compares the kernel
with, against the oracle's evaluation of the gate expansion `zkif-to-ir` produces for the same system
(fixtures.r1cs_to_gates, from_r1cs.rs:27-141): the first violated row of the whole system and, one row at a time, every
row's verdict.  The systems hold empty linear combinations, terms on variable 0, zero coefficients, C_r of several
general-coefficient terms, and assignments that satisfy them and that do not."""
import random

import numpy as np
import pytest

from oracle import evaluator as ev
from oracle import fixtures as fx
from oracle import r1cs as ro
from tests.util import FIELDS

N_PUBLIC = 3


def _le(v, p):
    return int(v).to_bytes((p.bit_length() + 7) // 8, "little")


def _csr(rows):
    """[[(col, coef_idx)] per row] -> (row_ptr, col, coef_idx)"""
    rp = np.zeros(len(rows) + 1, np.uint64)
    rp[1:] = np.cumsum([len(t) for t in rows])
    col = np.array([c for t in rows for c, _ in t], np.uint32)
    ci = np.array([i for t in rows for _, i in t], np.uint32)
    return rp, col, ci


def gate_expansion_first_failure(A, B, C, coefs, z, p, rows=None):
    """first violated row (-1: none) of the rows `rows` (default: all), by the oracle's evaluation of the gate expansion"""
    n_rows = len(A[0]) - 1
    rows = range(n_rows) if rows is None else rows
    cons = []
    for row in rows:
        cons.append(tuple([(int(col[e]), _le(coefs[int(ci[e])], p)) for e in range(int(rp[row]), int(rp[row + 1]))]
                          for rp, col, ci in (A, B, C)))
    instance_vars = [(i, _le(z[i], p)) for i in range(1, 1 + N_PUBLIC)]
    witness_ids = list(range(1 + N_PUBLIC, len(z)))
    msgs, _ = fx.r1cs_to_gates(_le(p - 1, p), instance_vars, witness_ids, cons, [_le(z[i], p) for i in witness_ids])
    tb = ev.TracingBackend()
    v = ev.Evaluator.from_messages(msgs, tb).get_violations()
    if not v:
        return -1
    assert v[0].startswith("Wire_")
    return len(tb.asserts) - 1          # one AssertZero per row, in row order: the failing one is the last reached


def small_system(p, seed, n_free=10, n_rows=18):
    """Row r: (A_r . z)(B_r . z) = C_r . z with C_r = rest_r + c_r z[s_r], s_r = n_free + 1 + r a slack read by no other
    row.  A_r, B_r, rest_r: 0 to 4 terms over variable 0 and the free variables, some with a zero coefficient.  Every
    fourth row has an empty C_r (then A_r or B_r is empty too, so that the row holds)."""
    rnd = random.Random(seed)
    coefs = [0, 1, p - 1] + [rnd.randrange(2, p - 1) for _ in range(6)]      # index 0: zero, 1: one
    n_vars = 1 + n_free + n_rows
    A, B, C = [], [], []
    for r in range(n_rows):
        def terms(k):
            return [(0 if rnd.random() < 0.25 else rnd.randrange(1, n_free + 1), rnd.randrange(len(coefs))) for _ in range(k)]
        a, b = terms(rnd.randrange(0, 5)), terms(rnd.randrange(0, 5))
        if r % 4 == 3:
            (a if r % 8 == 3 else b).clear()
            c = []
        else:
            c = terms(rnd.randrange(0, 4))
            c.insert(rnd.randrange(len(c) + 1), (n_free + 1 + r, rnd.randrange(2, len(coefs))))   # c_r != 0
        A.append(a), B.append(b), C.append(c)
    return _csr(A), _csr(B), _csr(C), coefs, n_vars


def satisfying(A, B, C, coefs, n_vars, n_free, p, seed):
    rnd = random.Random(seed)
    z = [1] + [rnd.randrange(p) for _ in range(n_free)] + [0] * (n_vars - 1 - n_free)
    for r in range(len(A[0]) - 1):
        rp, col, ci = C
        if rp[r] == rp[r + 1]:
            continue
        s = n_free + 1 + r
        slack_coef = next(coefs[int(ci[e])] for e in range(int(rp[r]), int(rp[r + 1])) if int(col[e]) == s)
        rest = ro.lc(C, r, coefs, z, p)                 # z[s] is still 0
        z[s] = (ro.lc(A, r, coefs, z, p) * ro.lc(B, r, coefs, z, p) - rest) * pow(slack_coef, -1, p) % p
    return z


@pytest.mark.parametrize("name", ["p101", "goldilocks", "bn254"])
def test_r1cs_reference_matches_gate_expansion(name):
    p = FIELDS[name]
    n_free = 10
    for seed in range(3):
        A, B, C, coefs, n_vars = small_system(p, seed, n_free=n_free)
        n_rows = len(A[0]) - 1
        good = satisfying(A, B, C, coefs, n_vars, n_free, p, seed)
        rnd = random.Random(100 + seed)
        zs = [good]
        slack_rows = [r for r in range(n_rows) if C[0][r] != C[0][r + 1]]
        for r in (slack_rows[0], slack_rows[len(slack_rows) // 2], slack_rows[-1]):
            bad = list(good)
            bad[n_free + 1 + r] = (bad[n_free + 1 + r] + rnd.randrange(1, p)) % p      # violates row r alone
            zs.append(bad)
            assert ro.row_verdicts(A, B, C, coefs, bad, p) == [x != r for x in range(n_rows)]
        bad = list(good)
        bad[1 + rnd.randrange(n_free)] = rnd.randrange(p)    # a free variable: every row that reads it may fail
        zs.append(bad)
        zs.append([1] + [rnd.randrange(p) for _ in range(n_vars - 1)])
        for z in zs:
            verdicts = ro.row_verdicts(A, B, C, coefs, z, p)
            first = ro.first_violated_row(A, B, C, coefs, z, p)
            assert first == (verdicts.index(False) if False in verdicts else -1)
            assert first == gate_expansion_first_failure(A, B, C, coefs, z, p)
            for r in range(n_rows):
                assert verdicts[r] == (gate_expansion_first_failure(A, B, C, coefs, z, p, rows=[r]) == -1), (name, seed, r)
        assert ro.first_violated_row(A, B, C, coefs, good, p) == -1
        # what the systems hold: empty LCs, terms on variable 0, zero coefficients, C_r of several general terms
        assert any(A[0][r] == A[0][r + 1] for r in range(n_rows)) and any(C[0][r] == C[0][r + 1] for r in range(n_rows))
        assert (np.concatenate([A[1], B[1], C[1]]) == 0).any() and (np.concatenate([A[2], B[2], C[2]]) == 0).any()
        assert any(sum(int(C[2][e]) >= 2 for e in range(int(C[0][r]), int(C[0][r + 1]))) >= 2 for r in range(n_rows))


def test_r1cs_reference_reduces_coefficients_and_values():
    """coefficients and values >= p act as their residues; an empty linear combination is 0"""
    p = FIELDS["p101"]
    A, B, C, coefs, n_vars = small_system(p, 7)
    z = satisfying(A, B, C, coefs, n_vars, 10, p, 7)
    lifted_coefs = [c + p * (i % 3) for i, c in enumerate(coefs)]
    lifted_z = [z[0]] + [v + 5 * p for v in z[1:]]
    assert ro.row_verdicts(A, B, C, lifted_coefs, lifted_z, p) == ro.row_verdicts(A, B, C, coefs, z, p)
    assert ro.first_violated_row(A, B, C, lifted_coefs, lifted_z, p) == -1
    assert ro.lc(A, next(r for r in range(len(A[0]) - 1) if A[0][r] == A[0][r + 1]), coefs, z, p) == 0
    assert ro.lc(_csr([[(1, 0), (2, 1)]]), 0, [p, 2 * p + 1], [1, 7, 9 + p], p) == 9
