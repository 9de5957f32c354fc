"""The R1CS check (`zkb_r1cs_*`, k_r1cs_check<N>) against the direct integer reference oracle/r1cs.py, at the shapes and
values where the kernel could go wrong without tests/test_gpu_r1cs.py noticing: every field width, worst-case lazy
accumulators, long rows up to the per-class limit, wide and ragged tiles, more rows than the grid has threads, sort
windows, raw values >= p and >= R, coefficient tables of any stride, and device-resident reuse.

The systems come from a structured generator: A_r and B_r read only variable 0 and free variables, and row r's slack
variable appears in C_r alone, so corrupting that slack violates row r and no other row.  Each assignment lane of a
batch can then target its own rows; its expected first failure is the smallest targeted row the reference finds
violated (the other rows hold, which the reference confirms once for the good assignment)."""
import random

import numpy as np
import pytest

from oracle import r1cs as ro
from tests.util import FIELDS, zkb

pytestmark = pytest.mark.gpu

ZERO, ONE, WORST = 0, 1, 2      # coefficient table: 0, 1, c* (c* R = p - 1 mod p), then general coefficients
N_GENERAL = 16


def nlimb(p):
    bits = p.bit_length()
    return 1 if bits <= 32 else 2 if bits <= 64 else 4 if bits <= 128 else 8


class System:
    """rows, coefficient table and a satisfying assignment `z` (reduced integers)"""

    def __init__(self, p, shapes, seed, n_free=48, extra_coefs=(), coef_stride=None):
        rnd = random.Random(seed)
        self.p, self.N = p, nlimb(p)
        self.eb = 4 * self.N
        self.R = 1 << (32 * self.N)
        self.Rinv = pow(self.R, -1, p)
        # worst case of the Montgomery domain: the kernel sums z R mod p and c R mod p; both are p - 1 for this value
        worst = (p - 1) * self.Rinv % p
        self.coefs = [0, 1, worst] + [rnd.randrange(2, p) for _ in range(N_GENERAL)] + list(extra_coefs)
        general = list(range(3, len(self.coefs))) + [WORST]
        cf = [c % p for c in self.coefs]
        assert all(cf[i] not in (0, 1) for i in general)
        self.n_free, self.n_rows = n_free, len(shapes)
        self.n_vars = 1 + n_free + self.n_rows
        n_worst = n_free // 2                       # variables 1 .. n_worst hold the worst-case value
        z = [1] + [worst] * n_worst + [rnd.randrange(p) for _ in range(n_free - n_worst)] + [0] * self.n_rows

        def term(kind):
            if kind == "mixed":
                kind = rnd.choice(["ones", "worst", "general", "general", "var0", "zero"])
            if kind == "ones":
                return rnd.randrange(1, n_worst + 1), ONE
            if kind == "worst":
                return rnd.randrange(1, n_worst + 1), WORST
            if kind == "general":
                return rnd.randrange(1, n_free + 1), rnd.choice(general)
            if kind == "var0":
                return 0, rnd.choice(general + [ONE])
            return rnd.randrange(0, n_free + 1), ZERO    # "zero": the term is dropped

        mats = ([], [], [])
        self.slack_coef = []
        for r, (kind, na, nb, nc, slack) in enumerate(shapes):
            a = [term(kind) for _ in range(na)]
            b = [term(kind) for _ in range(nb)]
            c = [term(kind) for _ in range(nc)]
            sc = ONE if slack == "one" else rnd.choice(general)
            c.insert(rnd.randrange(len(c) + 1), (self.slack_var(r), sc))
            lcv = [sum(cf[i] * z[v] for v, i in t) % p for t in (a, b, c)]       # z[slack] is still 0
            z[self.slack_var(r)] = (lcv[0] * lcv[1] - lcv[2]) * pow(cf[sc], -1, p) % p
            self.slack_coef.append(sc)
            for m, t in zip(mats, (a, b, c)):
                m.append(t)
        self.A, self.B, self.C = (self._csr(m) for m in mats)
        self.z = z
        cs = coef_stride or self.eb
        self.coef_table = np.stack([np.frombuffer(c.to_bytes(cs, "little"), np.uint8) for c in self.coefs])
        self.one_slack_rows = [r for r in range(self.n_rows) if self.slack_coef[r] == ONE]
        self._ab = {}

    @staticmethod
    def _csr(rows):
        rp = np.zeros(len(rows) + 1, np.uint64)
        rp[1:] = np.cumsum([len(t) for t in rows])
        col = np.array([v for t in rows for v, _ in t], np.uint32)
        ci = np.array([i for t in rows for _, i in t], np.uint32)
        return rp, col, ci

    def slack_var(self, row):
        return self.n_free + 1 + row

    def load(self, b):
        b.set_field(self.p)
        b.r1cs_load(self.A, self.B, self.C, self.coef_table, self.n_vars)

    def check_good(self):
        assert ro.first_violated_row(self.A, self.B, self.C, self.coefs, self.z, self.p) == -1

    # ---- lanes: a list of (row, raw value of that row's slack); a lane may also be a whole assignment (Full)
    def expected(self, lane):
        if isinstance(lane, Full):
            return ro.first_violated_row(self.A, self.B, self.C, self.coefs, lane.z, self.p)
        bad = []
        for row, v in lane:                 # a slack is read by its own C_r alone: A_r . z and B_r . z stay as they are
            if row not in self._ab:
                self._ab[row] = ro.lc(self.A, row, self.coefs, self.z, self.p) * ro.lc(self.B, row, self.coefs, self.z, self.p)
            s = self.slack_var(row)
            old, self.z[s] = self.z[s], v
            if (self._ab[row] - ro.lc(self.C, row, self.coefs, self.z, self.p)) % self.p:
                bad.append(row)
            self.z[s] = old
        return min(bad, default=-1)

    def batch(self, lanes, stride=None):
        """uint8 [len(lanes), n_vars, stride] of the lanes' raw values"""
        stride = stride or self.eb
        enc = lambda vals: np.frombuffer(b"".join(int(v).to_bytes(stride, "little") for v in vals), np.uint8).reshape(-1, stride)
        zb = np.repeat(enc(self.z)[None], len(lanes), axis=0)
        for j, lane in enumerate(lanes):
            if isinstance(lane, Full):
                zb[j] = enc(lane.z)
            else:
                for row, v in lane:
                    zb[j, self.slack_var(row)] = enc([v])[0]
        return zb

    # ---- raw slack values of a row: violations and congruent values
    def violations(self, row, wide=False, rnd=None):
        s, p = self.z[self.slack_var(row)], self.p
        out = [(s + (1 << (32 * j)) * self.Rinv) % p for j in range(self.N)]    # the stored residue differs in limb j
        out += [(s - 1) % p, p - s]
        if wide:
            k = self.big_multiple(rnd)
            out += [s + k * p + 1, s + k * p + (1 << (32 * (self.N - 1))) * self.Rinv % p]
        return out

    def congruent(self, row, wide=False, rnd=None):
        s, p = self.z[self.slack_var(row)], self.p
        out = [s + p] if s + p < self.R else []
        if wide:
            out += [s + p, s + self.big_multiple(rnd) * p, s + self.big_multiple(rnd) * p]
        return out

    def big_multiple(self, rnd):
        """k with k p >= R and s + k p below 2^64 R: a value >= R that fits a stride of element bytes + 8"""
        return rnd.randrange(self.R // self.p + 1, 1 << 63)

    def lifted(self, rnd):
        """every value but z_0 plus a multiple of p that puts it at or above R (stride element bytes + 8)"""
        return Full([self.z[0]] + [v + self.big_multiple(rnd) * self.p for v in self.z[1:]])


class Full:
    def __init__(self, z):
        self.z = z


def verdicts(v):
    return [(-1 if x["ok"] else int(x["first_fail_seq"])) for x in v]


def run_batch(b, S, lanes, stride=None):
    got = verdicts(b.r1cs_check(S.batch(lanes, stride)))
    exp = [S.expected(lane) for lane in lanes]
    bad = [(j, got[j], exp[j]) for j in range(len(lanes)) if got[j] != exp[j]]
    assert not bad, f"{len(bad)} of {len(lanes)} lanes differ (lane, kernel, reference): {bad[:12]}"
    return exp


def run_singly(b, S, lanes, stride=None):
    for j, lane in enumerate(lanes):
        b.r1cs_upload(S.batch([lane], stride))
        got, exp = verdicts(b.r1cs_run())[0], S.expected(lane)
        assert got == exp, (j, got, exp)


def mixed_shapes(rnd, n_rows, long_rows=()):
    """rows of 0, 1, 8 terms, all-ones, all-general, worst-case, mixed and all-zero-coefficient rows; C_r of several
    general terms with a general slack coefficient; plus `long_rows`; in random order"""
    base = [("ones", 0, 0, 0, "one"), ("general", 1, 1, 0, "one"), ("worst", 1, 1, 1, "general"),
            ("ones", 8, 8, 0, "one"), ("general", 8, 8, 3, "general"), ("mixed", 8, 8, 4, "general"),
            ("zero", 6, 6, 0, "one"), ("zero", 3, 5, 4, "general"), ("mixed", 0, 8, 2, "one"),
            ("general", 8, 0, 0, "one"), ("worst", 8, 8, 8, "one"), ("mixed", 1, 0, 5, "general")]
    shapes = [base[i % len(base)] for i in range(n_rows)] + list(long_rows)
    rnd.shuffle(shapes)
    return shapes


# long worst-case rows: the top accumulator limb overflows after ~2 terms at p256full, 5 at bls381, 28 at bn254 and
# ~450 at kat124; these rows pass that by 3x at kat124 and by far elsewhere, one of them at the per-class limit
LONG_ROWS = [("worst", 300, 300, 300, "general"), ("ones", 300, 300, 300, "one"), ("mixed", 300, 200, 100, "general"),
             ("worst", 1500, 1500, 1500, "one"), ("worst", 1500, 1500, 1500, "general"), ("worst", 65535, 1, 0, "one")]


def field_lanes(S, rnd, n, wide):
    """n lanes (0: only the targeted ones): each violation and congruent value of one row per lane (the limb-targeted
    ones on rows whose slack has coefficient one, so that the stored C_r . z differs in that limb alone), a few lanes
    with two targets, the rest good"""
    short = [r for r in range(S.n_rows) if S.A[0][r + 1] - S.A[0][r] < 1000]
    ones = [r for r in S.one_slack_rows if r in short]
    lanes = []
    for j, r in enumerate(rnd.sample(ones, S.N)):
        lanes.append([(r, S.violations(r)[j])])
    for v_idx in range(S.N, S.N + (4 if wide else 2)):
        r = rnd.choice(short)
        lanes.append([(r, S.violations(r, wide, rnd)[v_idx])])
    for r in rnd.sample(short, 4):
        lanes += [[(r, v)] for v in S.congruent(r, wide, rnd)]
    for _ in range(3):
        r1, r2 = sorted(rnd.sample(short, 2))
        lanes.append([(r2, S.violations(r2)[-2]), (r1, S.violations(r1)[0])])
    if wide:
        lanes.append(S.lifted(rnd))
    if n:
        assert len(lanes) <= n
        lanes += [[] for _ in range(n - len(lanes))]
    rnd.shuffle(lanes)
    return lanes


@pytest.fixture(scope="module")
def field_systems():
    cache = {}

    def get(name):
        if name not in cache:
            p = FIELDS[name]
            rnd = random.Random(p % 1000)
            S = System(p, mixed_shapes(rnd, 120, LONG_ROWS), seed=p % 997, n_free=64)
            S.check_good()
            cache[name] = S
        return cache[name]
    return get


@pytest.mark.parametrize("name", list(FIELDS))
def test_every_field_batch_of_70(name, field_systems, monkeypatch):
    """kind 1 (a tile of 128 lanes, 70 valid): element stride, then a stride of element bytes + 8 with values >= R"""
    monkeypatch.delenv("ZKB_TILE_LOG2", raising=False)
    S = field_systems(name)
    b = zkb().GpuBackend(0)
    S.load(b)
    rnd = random.Random(1)
    exp = run_batch(b, S, field_lanes(S, rnd, 70, wide=False))
    assert exp.count(-1) > 20 and sum(e != -1 for e in exp) >= S.N + 4
    run_batch(b, S, field_lanes(S, rnd, 70, wide=True), stride=S.eb + 8)
    assert b.timing()["level_launches"] == 1


@pytest.mark.parametrize("name", list(FIELDS))
def test_every_field_one_assignment(name, field_systems):
    """kind 0: the same violations and congruent values, one assignment per run"""
    S = field_systems(name)
    b = zkb().GpuBackend(0)
    S.load(b)
    rnd = random.Random(2)
    run_singly(b, S, field_lanes(S, rnd, 0, wide=False) + [[]])
    wide = [lane for lane in field_lanes(S, rnd, 0, wide=True) if isinstance(lane, Full) or
            any(v >= S.R for _, v in lane)] + [[]]
    run_singly(b, S, wide, stride=S.eb + 8)


TARGET_LANES = [0, 31, 32, 255, 256, 511, 512, 1023, 1024]


@pytest.mark.parametrize("n,tile_log2,tiles", [(1, None, 1), (8, "3", 1), (96, "5", 3), (300, None, 1), (1100, "10", 2)])
def test_tile_widths(n, tile_log2, tiles, monkeypatch):
    """1 lane; 8 (kind 0 over one tile of 8); 3 tiles of 32 (kind 1 over several tiles); 300 (one ragged tile of 512:
    a grid stride of two CTAs); 1100 (two tiles of 1024: four CTAs).  Targeted lanes at the warp, CTA and tile edges"""
    if tile_log2 is None:
        monkeypatch.delenv("ZKB_TILE_LOG2", raising=False)
    else:
        monkeypatch.setenv("ZKB_TILE_LOG2", tile_log2)
    p = FIELDS["bn254"]
    rnd = random.Random(n)
    S = System(p, mixed_shapes(rnd, 260), seed=n, n_free=40)
    S.check_good()
    b = zkb().GpuBackend(0)
    S.load(b)
    lanes = [[] for _ in range(n)]
    targets = sorted({j for j in TARGET_LANES if j < n} | {n - 1})
    rows = rnd.sample(range(S.n_rows), len(targets))
    for j, r in zip(targets, rows):
        lanes[j] = [(r, rnd.choice(S.violations(r)))]
    exp = run_batch(b, S, lanes)
    assert sum(e != -1 for e in exp) >= len(targets) - 1
    assert b.timing()["level_launches"] == tiles


def test_more_rows_than_threads_across_the_sort_window():
    """262144 + 4000 rows, one assignment: every thread walks several rows, and the second kind-0 sort window holds
    the violated rows"""
    p = FIELDS["bn254"]
    rnd = random.Random(5)
    kinds = [("general", 1, 1, 0, "one"), ("mixed", 2, 1, 1, "general"), ("ones", 3, 2, 0, "one"), ("worst", 1, 2, 0, "one")]
    shapes = [kinds[rnd.randrange(len(kinds))] for _ in range(262144 + 4000)]
    S = System(p, shapes, seed=5, n_free=200)
    S.check_good()
    b = zkb().GpuBackend(0)
    S.load(b)
    w2 = 262144
    lanes = [[], [(w2 + 1234, S.violations(w2 + 1234)[0])], [(S.n_rows - 1, S.violations(S.n_rows - 1)[7])],
             [(w2 + 3000, S.violations(w2 + 3000)[-1]), (w2 + 17, S.violations(w2 + 17)[3])],
             [(w2 + 5, S.congruent(w2 + 5)[0])], []]
    run_singly(b, S, lanes)


def test_small_sort_windows(monkeypatch):
    """ZKB_R1CS_SIGMA=64 on 2000 rows of varied length, both layout kinds: targeted rows in many windows"""
    monkeypatch.setenv("ZKB_R1CS_SIGMA", "64")
    monkeypatch.delenv("ZKB_TILE_LOG2", raising=False)
    p = FIELDS["goldilocks"]
    rnd = random.Random(6)
    shapes = []
    for _ in range(2000):
        shapes.append((rnd.choice(["ones", "general", "mixed", "worst"]), rnd.randrange(0, 12), rnd.randrange(0, 12),
                       rnd.randrange(0, 4), rnd.choice(["one", "general"])))
    S = System(p, shapes, seed=6)
    S.check_good()
    b = zkb().GpuBackend(0)
    S.load(b)
    windows = rnd.sample(range(2000 // 64), 24)
    lanes = []
    for w in windows:
        r = w * 64 + rnd.randrange(64)
        lanes.append([(r, rnd.choice(S.violations(r)))])
    for i in range(0, 12, 2):              # two targets in different windows: the smaller row is reported
        lanes.append(lanes[i] + lanes[i + 1])
    lanes += [[] for _ in range(10)]
    run_batch(b, S, lanes)                 # kind 1
    run_singly(b, S, lanes[::3] + [lanes[-1]])  # kind 0


def limit_system(n_terms, seed=7, p=FIELDS["bls381"]):
    rnd = random.Random(seed)
    shapes = mixed_shapes(rnd, 40)
    shapes.insert(7, ("worst", n_terms, 2, 1, "one"))
    return System(p, shapes, seed=seed)


def test_per_class_limit():
    """one linear combination of exactly 65535 general terms checks in both kinds; 65536 is rejected"""
    S = limit_system(65535)
    S.check_good()
    b = zkb().GpuBackend(0)
    S.load(b)
    lanes = [[], [(7, S.violations(7)[0])], [(7, S.violations(7)[S.N - 1])], [(7, S.congruent(7)[0])],
             [(20, S.violations(20)[1])], [(30, S.violations(30)[2]), (7, S.violations(7)[-1])]]
    run_singly(b, S, lanes)
    run_batch(b, S, lanes * 6 + [[]] * 4)
    z_ = zkb()
    T = limit_system(65536)
    b2 = z_.GpuBackend(0)
    T.load(b2)
    for n in (1, 40):
        with pytest.raises(z_.ZkbError) as e:
            b2.r1cs_check(T.batch([[]] * n))
        assert e.value.code == z_.ZKB_E_UNSUPPORTED


@pytest.mark.parametrize("n_rows", [0, 1, 31, 32, 33])
def test_row_counts(n_rows):
    """no rows (every verdict true), one row, and one slice with no, one and 31 padding rows, in both kinds"""
    p = FIELDS["kat124"]
    rnd = random.Random(n_rows)
    S = System(p, mixed_shapes(rnd, n_rows), seed=n_rows, n_free=12)
    S.check_good()
    b = zkb().GpuBackend(0)
    S.load(b)
    lanes = [[]] + [[(r, S.violations(r)[r % (S.N + 2)])] for r in range(n_rows)]
    if n_rows:
        lanes.append([(n_rows - 1, S.violations(n_rows - 1)[-1])])
    run_singly(b, S, lanes[:1] + lanes[-3:])
    lanes = (lanes * (40 // len(lanes) + 1))[:40]
    exp = run_batch(b, S, lanes)
    assert n_rows or exp == [-1] * 40


def test_device_resident_reuse(monkeypatch):
    """one context: 1 -> 70 -> 1 assignments (both layouts built once and kept), then another system on it"""
    monkeypatch.delenv("ZKB_TILE_LOG2", raising=False)
    p = FIELDS["bls381"]
    rnd = random.Random(9)
    S = System(p, mixed_shapes(rnd, 150, LONG_ROWS[:2]), seed=9)
    S.check_good()
    b = zkb().GpuBackend(0)
    S.load(b)
    lanes = field_lanes(S, rnd, 70, wide=False)
    hit = next(j for j, lane in enumerate(lanes) if lane and S.expected(lane) != -1)

    def single(lane, system):
        b.r1cs_upload(system.batch([lane]))
        assert verdicts(b.r1cs_run()) == [system.expected(lane)]

    single(lanes[hit], S)
    b.r1cs_upload(S.batch(lanes))
    assert verdicts(b.r1cs_run()) == [S.expected(lane) for lane in lanes]
    single([], S)
    single(lanes[hit], S)
    T = System(p, mixed_shapes(rnd, 90), seed=10, n_free=20)
    T.check_good()
    T.load(b)
    other = field_lanes(T, rnd, 70, wide=False)
    b.r1cs_upload(T.batch(other))
    assert verdicts(b.r1cs_run()) == [T.expected(lane) for lane in other]
    single(next(lane for lane in other if lane and T.expected(lane) != -1), T)


@pytest.mark.parametrize("name", ["goldilocks", "bn254", "p256full"])
def test_coefficient_table_wide_entries(name, monkeypatch):
    """table entries of element bytes + 8: p (the term is dropped), 2p + 1 (coefficient one), general + p, general + k p
    >= R and c* + p, used in every row shape, in both kinds"""
    monkeypatch.delenv("ZKB_TILE_LOG2", raising=False)
    p = FIELDS[name]
    rnd = random.Random(11)
    R = 1 << (32 * nlimb(p))
    g = rnd.randrange(2, p)
    worst = (p - 1) * pow(R, -1, p) % p
    extra = [g + p, g + rnd.randrange(R // p + 1, 1 << 63) * p, worst + p]
    S = System(p, mixed_shapes(rnd, 120), seed=11, extra_coefs=extra, coef_stride=nlimb(p) * 4 + 8)
    # re-point the zero and one terms at the entries p and 2p + 1: the same classes, other bytes
    S.coefs += [p, 2 * p + 1]
    S.coef_table = np.stack([np.frombuffer(c.to_bytes(nlimb(p) * 4 + 8, "little"), np.uint8) for c in S.coefs])
    for _, _, ci in (S.A, S.B, S.C):
        ci[ci == ZERO] = len(S.coefs) - 2
        ci[ci == ONE] = len(S.coefs) - 1
    S.check_good()
    b = zkb().GpuBackend(0)
    S.load(b)
    lanes = field_lanes(S, rnd, 50, wide=False)
    run_batch(b, S, lanes)
    run_singly(b, S, [lane for lane in lanes if lane][:8] + [[]])


def test_failed_upload_leaves_nothing_to_run(monkeypatch):
    """a row of 40000 ones + 40000 general terms in A checks with one assignment (kind 0 counts them as two classes)
    and is rejected at >= 32 (kind 1: one class per matrix); the rejected upload must not leave the previous geometry
    over the new bytes: the next run fails until an upload succeeds"""
    monkeypatch.delenv("ZKB_TILE_LOG2", raising=False)
    z_ = zkb()
    p = FIELDS["bn254"]
    rnd = random.Random(12)
    S = System(p, mixed_shapes(rnd, 20), seed=12)
    # row 3 of A: 40000 coefficient-one terms + 40000 general terms
    rp, col, ci = S.A
    r0 = int(rp[4])
    extra_cols = np.array([rnd.randrange(1, S.n_free + 1) for _ in range(80000)], np.uint32)
    extra_ci = np.array([ONE] * 40000 + [WORST] * 40000, np.uint32)
    S.A = (np.concatenate([rp[:4], rp[4:] + 80000]).astype(np.uint64),
           np.concatenate([col[:r0], extra_cols, col[r0:]]), np.concatenate([ci[:r0], extra_ci, ci[r0:]]))
    # re-solve row 3's slack for its longer A_r
    s = S.slack_var(3)
    S.z[s] = 0
    rhs = ro.lc(S.A, 3, S.coefs, S.z, p) * ro.lc(S.B, 3, S.coefs, S.z, p) - ro.lc(S.C, 3, S.coefs, S.z, p)
    S.z[s] = rhs * pow(S.coefs[S.slack_coef[3]] % p, -1, p) % p
    S.check_good()
    b = z_.GpuBackend(0)
    S.load(b)
    bad = [(3, S.violations(3)[0])]
    b.r1cs_upload(S.batch([bad]))
    assert verdicts(b.r1cs_run()) == [3]
    with pytest.raises(z_.ZkbError) as e:
        b.r1cs_upload(S.batch([[]] * 64))
    assert e.value.code == z_.ZKB_E_UNSUPPORTED
    with pytest.raises(z_.ZkbError) as e:
        b.r1cs_run()
    assert e.value.code == z_.ZKB_E_ARG
    b.r1cs_upload(S.batch([[]]))
    assert verdicts(b.r1cs_run()) == [-1]
    b.r1cs_upload(S.batch([bad]))
    assert verdicts(b.r1cs_run()) == [3]
