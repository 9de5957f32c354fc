"""R1CS satisfiability in plain Python integers — TEST INFRASTRUCTURE ONLY.

The check `zkb_r1cs_*` computes, stated directly:  row r holds when
    (A_r . z) (B_r . z) - (C_r . z) == 0  (mod p),
with every matrix in the project's CSR form `(row_ptr, col, coef_idx)` and `coefs` the coefficient table as integers.
Coefficients and values are reduced mod p (a table entry or a value may be >= p); an empty linear combination is 0.
This is what the gate expansion of `from_r1cs.rs:71-125` evaluates (pinned by tests/test_oracle_r1cs.py), without its
cost, so tests can check systems of hundreds of thousands of rows or rows of 65535 terms.
"""
from __future__ import annotations


def _lists(M):
    rp, col, ci = M
    return [int(x) for x in rp], [int(x) for x in col], [int(x) for x in ci]


def lc(M, row: int, coefs, z, p: int) -> int:
    """sum over the terms of row `row` of M of coefs[ci] * z[col], mod p"""
    rp, col, ci = M
    s = 0
    for e in range(int(rp[row]), int(rp[row + 1])):
        s += int(coefs[int(ci[e])]) % p * (int(z[int(col[e])]) % p)
    return s % p


def row_verdicts(A, B, C, coefs, z, p: int) -> list:
    """[bool] per row: True when (A_r . z)(B_r . z) == C_r . z (mod p)"""
    cf = [int(c) % p for c in coefs]
    zz = [int(v) % p for v in z]
    mats = [_lists(M) for M in (A, B, C)]
    n_rows = len(mats[0][0]) - 1
    out = []
    for row in range(n_rows):
        v = []
        for rp, col, ci in mats:
            s = 0
            for e in range(rp[row], rp[row + 1]):
                s += cf[ci[e]] * zz[col[e]]
            v.append(s % p)
        out.append((v[0] * v[1] - v[2]) % p == 0)
    return out


def first_violated_row(A, B, C, coefs, z, p: int) -> int:
    """-1 when every row holds, else the smallest violated (original) row"""
    for row, ok in enumerate(row_verdicts(A, B, C, coefs, z, p)):
        if not ok:
            return row
    return -1
