"""Value sets on the device: every set of a batch must give what the oracle's `evaluate` gives for that set's own statement
(an OraclePanic is status ZKB_E_FATAL), on one context, on several contexts of one device, and through `zkb evaluate --sets`."""
import os
import subprocess

import numpy as np
import pytest

from oracle import evaluator as ev
from oracle import ir
from oracle import sieve_fbs as F
from tests.gen_programs import Gen
from tests.test_value_sets_host import BLS, make_sets, record_batch, set_statement
from tests.util import ROOT, zkb

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "zkinterface-ir_b200", "zkb")
WORKSPACES = ["example", "example_incorrect", "boolean_example", "boolean_example_incorrect", "builder_switch",
              "builder_switch_nested", "r1cs_example"]


def oracle_result(msgs):
    try:
        return 0, ev.evaluate(msgs)
    except ir.OraclePanic as p:
        return zkb().ZKB_E_FATAL, [str(p)]


def n_devices():
    import torch
    return torch.cuda.device_count()


def read_ws(ws):
    msgs = []
    for fn in ("000_instance.sieve", "001_witness.sieve", "002_relation.sieve"):
        msgs += F.read_messages(open(os.path.join(GOLDEN, ws, fn), "rb").read())
    inst = [v for m in msgs if isinstance(m, ir.Instance) for v in m.common_inputs]
    wit = [v for m in msgs if isinstance(m, ir.Witness) for v in m.short_witness]
    rels = [m for m in msgs if isinstance(m, ir.Relation)]
    return inst, wit, rels


def golden_sets(ws):
    """the workspace's own values, a wrong witness value, short instance / witness streams, an assertion failing before the
    witness stream runs out, and raw witness values >= p"""
    inst, wit, rels = read_ws(ws)
    p = int.from_bytes(rels[0].header.field_characteristic, "little")
    num = [int.from_bytes(v, "little") for v in wit]

    def le(xs):
        return [ir.le_bytes(x) for x in xs]
    sets = [(inst, wit)]
    for k in range(len(wit)):
        sets.append((inst, le(num[:k] + [(num[k] + 1) % p] + num[k + 1:])))   # one wrong value
        sets.append((inst, wit[:k]))                                           # short witness stream
        sets.append((inst, le(num[:k] + [(num[k] + 1) % p]) + wit[k + 1:-1]))  # wrong value, then too few
        sets.append((inst, le(num[:k] + [num[k] + p] + num[k + 1:])))          # raw value >= p
    for k in range(len(inst)):
        sets.append((inst[:k], wit))                                           # short instance stream
    return rels, sets


@pytest.mark.parametrize("ws", WORKSPACES)
def test_golden_workspaces_split_into_sets(ws):
    z = zkb()
    rels, sets = golden_sets(ws)
    h = rels[0].header
    e = z.Evaluator(z.GpuBackend(0))
    for si, sw in sets:
        e.add_value_set(z.Source.from_buffers([F.write_messages([ir.Instance(h, si), ir.Witness(h, sw)])]))
    e.ingest_source(z.Source.from_buffers([F.write_messages(rels)]))
    got = e.get_batch_violations()
    statuses = set()
    for j, (si, sw) in enumerate(sets):
        want = oracle_result([ir.Instance(h, si), ir.Witness(h, sw)] + rels)
        assert got[j] == want, (ws, j, got[j], want)
        statuses.add((want[0], bool(want[1])))
    assert len(statuses) >= 2, statuses


CASES = [(seed, 101, False, 40) for seed in range(8)] + [(seed, 2, True, 40) for seed in range(100, 104)] + \
        [(seed, (1 << 64) - (1 << 32) + 1, False, 40) for seed in range(200, 203)] + [(300, BLS, False, 40), (301, BLS, False, 300)]


@pytest.mark.parametrize("seed,p,boolean,n_sets", CASES)
def test_random_programs_against_the_oracle(seed, p, boolean, n_sets, monkeypatch):
    monkeypatch.setenv("ZKB_TILE_LOG2", "5")   # 32 witnesses per tile: sets cross tile boundaries
    z = zkb()
    msgs = Gen(seed, p, boolean).statement()
    h = msgs[2].header
    ci, cw, sets = make_sets(seed, msgs, n_sets)
    e = record_batch(z, h, ci, cw, sets, msgs[2], backend=z.GpuBackend(0))
    got = e.get_batch_violations()
    for j, s in enumerate(sets):
        assert got[j] == oracle_result(set_statement(h, (ci, cw), s, msgs[2])), j


@pytest.mark.parametrize("seed,p,boolean", [(1, 101, False), (3, 101, False), (101, 2, True), (201, (1 << 64) - (1 << 32) + 1, False)])
def test_sets_differing_only_in_instances_and_common_instances(seed, p, boolean):
    z = zkb()
    msgs = Gen(seed, p, boolean).statement()
    h = msgs[2].header
    inst, wit = list(msgs[0].common_inputs), list(msgs[1].short_witness)
    rng = np.random.default_rng(seed)

    def rv(n):
        return [ir.le_bytes(int(rng.integers(0, min(p, 1 << 40)))) for _ in range(n)]
    for common, sets in ((([], wit), [(rv(len(inst)), []) for _ in range(50)]),          # witness common, instances per set
                         ((inst, []), [([], rv(len(wit) - k % 3)) for k in range(50)])):  # instance common, own witnesses
        e = record_batch(z, h, common[0], common[1], sets, msgs[2], backend=z.GpuBackend(0))
        got = e.get_batch_violations()
        for j, s in enumerate(sets):
            assert got[j] == oracle_result(set_statement(h, common, s, msgs[2])), j


def test_get_of_and_capture_against_oracle_values():
    z = zkb()
    for seed, p, boolean in ((5, 101, False), (102, 2, True), (300, BLS, False)):
        msgs = Gen(seed, p, boolean).statement()
        h = msgs[2].header
        ci, cw, sets = make_sets(seed, msgs, 70)
        e = record_batch(z, h, ci, cw, sets, msgs[2], backend=z.GpuBackend(0))
        got = e.get_batch_violations()
        wires = None
        checked = 0
        for j, s in enumerate(sets):
            tb = ev.TracingBackend()
            try:
                o = ev.Evaluator.from_messages(set_statement(h, (ci, cw), s, msgs[2]), tb)
                viol = o.get_violations()
            except ir.OraclePanic:
                continue
            if viol:
                continue
            vals = {wid: w[1] for wid, w in o.values.items()}
            for wid, v in vals.items():
                assert e.get_of(j, wid) == v, (seed, j, wid)
            if wires is None and vals:
                wires = sorted(vals)
                e.capture_wires(wires)
                cap = e.backend.read_captured()
                assert cap.shape[0] == len(sets)
            if wires is not None and all(w in vals for w in wires):
                assert [int.from_bytes(cap[j, i].tobytes(), "little") for i in range(len(wires))] == [vals[w] for w in wires]
                checked += 1
        assert got and checked >= 1, seed


def test_batch_of_one_equals_get_violations():
    z = zkb()
    for ws in WORKSPACES:
        rels, sets = golden_sets(ws)
        h = rels[0].header
        for si, sw in sets[:6]:
            e = z.Evaluator(z.GpuBackend(0))
            e.add_value_set(z.Source.from_buffers([F.write_messages([ir.Instance(h, si), ir.Witness(h, sw)])]))
            e.ingest_source(z.Source.from_buffers([F.write_messages(rels)]))
            one = z.Evaluator(z.GpuBackend(0))
            try:
                one.ingest_source(z.Source.from_buffers([F.write_messages([ir.Instance(h, si), ir.Witness(h, sw)] + rels)]))
                single = (0, one.get_violations())
            except z.ZkbError as err:
                single = (err.code, [str(err)])
            assert e.get_batch_violations() == [single], ws


def run_sharded(z, devices, h, ci, cw, sets, rel):
    sb = z.ShardedBackend(devices)
    e = record_batch(z, h, ci, cw, sets, rel, backend=sb.root)
    e.use_devices(sb)
    return sb, e, e.get_batch_violations()


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0], "multi"])
def test_sharded_equals_single_context(devices, monkeypatch):
    if devices == "multi":
        if n_devices() < 2:
            pytest.skip("needs two devices (NCCL transport)")
        devices = list(range(n_devices()))
    monkeypatch.setenv("ZKB_TILE_LOG2", "5")
    z = zkb()
    for seed, p, boolean, n in ((7, 101, False, 150), (103, 2, True, 70), (300, BLS, False, 2)):
        msgs = Gen(seed, p, boolean).statement()
        h = msgs[2].header
        ci, cw, sets = make_sets(seed, msgs, n)
        single = record_batch(z, h, ci, cw, sets, msgs[2], backend=z.GpuBackend(0))
        want = single.get_batch_violations()
        sb, e, got = run_sharded(z, devices, h, ci, cw, sets, msgs[2])
        assert got == want, seed
        ok = [j for j, (st, v) in enumerate(want) if st == 0 and not v]
        if ok:
            wid = max(single_wires(msgs, h, ci, cw, sets[ok[-1]]), default=None)
            if wid is not None:
                assert e.get_of(ok[-1], wid) == single.get_of(ok[-1], wid)
        sb.close()


def single_wires(msgs, h, ci, cw, s):
    o = ev.Evaluator.from_messages(set_statement(h, (ci, cw), s, msgs[2]), ev.PlaintextBackend())
    return list(o.values)


def write_sets(tmp_path, ws):
    rels, sets = golden_sets(ws)
    h = rels[0].header
    (tmp_path / "rel").mkdir()
    (tmp_path / "rel" / "002_relation.sieve").write_bytes(F.write_messages(rels))
    names = []
    for j, (si, sw) in enumerate(sets):
        d = tmp_path / "sets" / f"set{j:03d}"
        d.mkdir(parents=True)
        (d / "000_instance.sieve").write_bytes(F.write_messages([ir.Instance(h, si)]))
        (d / "001_witness.sieve").write_bytes(F.write_messages([ir.Witness(h, sw)]))
        names.append(d.name)
    return names


def cli(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, timeout=300)


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_cli_sets(tmp_path, devices):
    names = write_sets(tmp_path, "example")
    extra = ["--devices", devices] if devices else []
    r = cli("evaluate", *extra, "--sets", str(tmp_path / "sets"), str(tmp_path / "rel"))
    want, n_bad = "", 0
    for name in names:
        one = cli("evaluate", str(tmp_path / "rel"), str(tmp_path / "sets" / name))
        want += f"== {name} ==\n" + one.stderr
        n_bad += one.returncode != 0
    assert 0 < n_bad < len(names)
    assert r.stderr == want + f"Error: {n_bad} of {len(names)} statements are NOT TRUE.\n"
    assert r.returncode == 1


def test_cli_sets_all_true_and_relation_in_a_set(tmp_path):
    names = write_sets(tmp_path, "builder_switch")
    import shutil
    for name in names[1:]:
        shutil.rmtree(tmp_path / "sets" / name)
    r = cli("evaluate", "--sets", str(tmp_path / "sets"), str(tmp_path / "rel"))
    assert r.returncode == 0, r.stderr
    assert r.stderr == f"== {names[0]} ==\n\nThe statement is TRUE!\n"
    shutil.copy(tmp_path / "rel" / "002_relation.sieve", tmp_path / "sets" / names[0] / "002_relation.sieve")
    r = cli("evaluate", "--sets", str(tmp_path / "sets"), str(tmp_path / "rel"))
    assert r.returncode == 1 and "002_relation.sieve" in r.stderr and r.stderr.startswith("Error: ")


def test_cpp_mirror(tmp_path):
    src = os.path.join(ROOT, "tests", "native", "value_sets_api.cpp")
    pkg = os.path.join(ROOT, "zkinterface-ir_b200")
    exe = str(tmp_path / "value_sets_api")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", exe, "-L", pkg, "-lzkb",
                           f"-Wl,-rpath,{pkg}"])
    r = subprocess.run([exe, GOLDEN], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == "value_sets_api ok"


def test_get_of_refuses_a_set_that_stops_early():
    """wire 2 is freed at the end of the relation: a set whose instance stream runs out stops before, where its own scope
    still holds wire 2, so its wires are not answered from the final scope"""
    z = zkb()
    from oracle import fixtures as fx
    h = fx.example_header()
    rel = ir.Relation(h, ir.ARITH, ir.SIMPLE, [], [
        ("Witness", 0), ("Add", 2, 0, 0), ("Instance", 1), ("Witness", 3), ("Free", 2, None)])
    lit = ir.literal32
    sets = [([lit(5)], [lit(7), lit(9)]), ([], [lit(7), lit(9)])]
    e = record_batch(z, h, [], [], sets, rel, backend=z.GpuBackend(0))
    got = e.get_batch_violations()
    assert got == [oracle_result(set_statement(h, ([], []), s, rel)) for s in sets]
    assert got[1] == (0, ["Not enough instance to consume"])
    assert e.get_of(0, 0) == 7 and e.get_of(0, 3) == 9
    with pytest.raises(z.ZkbError) as err:
        e.get_of(0, 2)
    assert err.value.code == z.ZKB_E_SEMANTIC
    with pytest.raises(z.ZkbError) as err:
        e.get_of(1, 2)
    assert err.value.code == z.ZKB_E_ARG and "stops recording" in str(err.value)
