"""Capture list on the device (zkb_capture_values / zkb_read_captured, kernels.cu: k_capture / k_bool_capture).

For every case the captured array equals zkb_read_values for every witness and value, byte for byte, and the oracle on
sampled witnesses: 1-, 2-, 4- and 8-limb fields and p = 2, ragged batches over small tiles, each execution path (per
wavefront, cooperative / cluster, the one-witness dataflow launch, Boolean CTA runs), sinks captured on tiles that skip
their sink stores, raw inputs and constants >= p, call-group outputs, two sharded contexts and the zkb.hpp mirror.  A list
changes neither the verdicts nor, once cleared, the stores and launches of a run."""
import os
import subprocess

import numpy as np
import pytest

from oracle import evaluator as ev
from oracle import flat
from tests.util import FIELDS, ROOT, circuits, random_flat_program, zkb

pytestmark = pytest.mark.gpu

PRIME_FIELDS = {"m31": 1, "goldilocks": 2, "kat124": 4, "bls381": 8}   # field -> limbs


def as_ints(rows):
    return [int.from_bytes(r.tobytes(), "little") for r in rows]


def check_against_read_values(b, handles, n_batch, stride):
    cap = b.read_captured(0, n_batch, stride)
    assert cap.shape == (n_batch, len(handles), stride)
    for j in range(n_batch):
        assert as_ints(cap[j]) == b.read_values(j, handles, stride), j
    return cap


def live_wires(b, n_wires):
    out = []
    for w in range(n_wires):
        try:
            out.append((w, b.scope_lookup(w)))
        except zkb().ZkbError:
            pass
    return out


def run_random(field, n_batch, env, monkeypatch, n_gates=1 << 12):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = circuits()
    z = zkb()
    p = FIELDS[field]
    eb = c.elem_bytes(p)
    circ = c.random_circuit(n_gates, 32, p, seed=11, n_tracked=8)
    wit = c.make_witnesses(circ, n_batch, seed=5, corrupt={n_batch // 2: 3} if n_batch > 2 else {})
    b = z.GpuBackend(0)
    b.set_field(p)
    b.push_gates(circ.gates, circ.const_pool)
    b.finalize()
    assert b.stats()["n_sink_ops"] > 0
    v0 = b.evaluate(None, wit, n_batch)
    launches0 = b.timing()["kernel_launches"]
    live = live_wires(b, circ.n_wires)
    handles = [h for _, h in live]
    b.capture(handles)
    v1 = b.run()
    assert np.array_equal(v0, v1)
    cap = check_against_read_values(b, handles, n_batch, eb)
    # the oracle, on the first, a middle and the last satisfied witness
    good = [j for j in range(n_batch) if v1[j]["ok"]]
    for j in sorted(set([good[0], good[len(good) // 2], good[-1]])):
        _, dump = flat.eval_dump(circ.gates, circ.const_pool, p.to_bytes(eb, "little"), None, wit[j], circ.n_wires, stride=eb)
        assert as_ints(cap[j]) == as_ints(dump[[w for w, _ in live]]), j
    # clearing the list gives the run back its skipped stores and its launches
    b.capture([])
    v2 = b.run()
    assert np.array_equal(v0, v2) and b.timing()["kernel_launches"] == launches0
    with pytest.raises(z.ZkbError):
        b.read_captured(0, 1, eb)
    b.close()


@pytest.mark.parametrize("path", ["wavefront", "coop"])
@pytest.mark.parametrize("n_batch", [1, 255, 257, 1000])
@pytest.mark.parametrize("field", list(PRIME_FIELDS))
def test_gpu_capture_prime_fields(field, n_batch, path, monkeypatch):
    env = {"ZKB_TILE_LOG2": "6"}
    if path == "wavefront":
        env["ZKB_COOP"] = "0"
    run_random(field, n_batch, env, monkeypatch)


@pytest.mark.parametrize("field", ["m31", "goldilocks"])
def test_gpu_capture_dataflow_launch(field, monkeypatch):
    """one-witness tiles of a 1- / 2-limb field: every tile is one k_levels_flow launch"""
    run_random(field, 5, {"ZKB_TILE_LOG2": "0", "ZKB_FLOW_MIN": "1"}, monkeypatch)


@pytest.mark.parametrize("n_batch", [1, 100, 257])
def test_gpu_capture_boolean(n_batch, monkeypatch):
    """p = 2 over 32-witness tiles (Boolean CTA runs), raw inputs >= 2 included"""
    monkeypatch.setenv("ZKB_TILE_LOG2", "5")
    z = zkb()
    gates, pool, n_wires = random_flat_program(2, 1500, 3, 6, seed=9, bool_ops=True)
    rng = np.random.default_rng(n_batch)
    inst = rng.integers(0, 2, size=(n_batch, 3, 1)).astype(np.uint8)
    wit = rng.integers(0, 2, size=(n_batch, 6, 1)).astype(np.uint8)
    wit[::3, 0, 0] = 3   # raw values >= p: read back unreduced
    b = z.GpuBackend(0)
    b.set_field(2, is_boolean=True)
    b.push_gates(gates, pool)
    b.finalize(keep_all_values=True)
    handles = list(range(b.stats()["n_values"]))
    v0 = b.evaluate(inst, wit, n_batch)
    b.capture(handles)
    assert np.array_equal(b.run(), v0)
    cap = check_against_read_values(b, handles, n_batch, 4)
    assert (cap[::3, 3 + 0, 0] == 3).all()   # value 3 is witness 0
    ref = flat.eval_batch(gates, pool, b"\x02", inst, wit, n_batch)
    assert [bool(x["ok"]) for x in v0] == [int(r["status"]) == flat.EV_TRUE for r in ref]
    b.close()


@pytest.mark.parametrize("field", list(PRIME_FIELDS))
def test_gpu_capture_raw_inputs_and_constants(field):
    """instance / witness values >= p and a constant >= p come back raw, as zkb_read_values returns them"""
    c = circuits()
    z = zkb()
    p = FIELDS[field]
    eb = c.elem_bytes(p)
    stride = eb + 8
    big = p + 12345
    pool = np.stack([c.le_bytes(big, stride), c.le_bytes(7, stride)])
    G = [(c.G_INSTANCE, 0, 0, 0), (c.G_WITNESS, 1, 0, 0), (c.G_CONSTANT, 2, 0, 0), (c.G_CONSTANT, 3, 0, 1),
         (c.G_ADD, 4, 0, 1), (c.G_MUL, 5, 4, 2), (c.G_ADD_CONSTANT, 6, 5, 1)]
    gates = np.array([(op, (0, 0, 0), out, a, bb) for op, out, a, bb in G], dtype=z.GATE_DTYPE)
    n_batch = 70
    rng = np.random.default_rng(1)
    ivals = [int(x) for x in rng.integers(0, 1 << 60, n_batch)]
    ivals[::4] = [p + k for k in range(len(ivals[::4]))]
    ivals[1] = (1 << (8 * eb)) + 5   # wider than an element
    wvals = [(p - 1 - k) if k % 3 else (2 * p + k) for k in range(n_batch)]
    inst = np.stack([c.le_bytes(x, stride) for x in ivals])[:, None, :]
    wit = np.stack([c.le_bytes(x, stride) for x in wvals])[:, None, :]
    b = z.GpuBackend(0)
    b.set_field(p)
    b.push_gates(gates, pool)
    b.finalize(keep_all_values=True)
    handles = [b.scope_lookup(w) for w in range(7)]
    b.capture(handles)
    b.evaluate(inst, wit, n_batch)
    cap = check_against_read_values(b, handles, n_batch, stride)
    for j in range(n_batch):
        s = (ivals[j] + wvals[j]) % p
        assert as_ints(cap[j]) == [ivals[j], wvals[j], big, 7, s, s * big % p, (s * big + 7) % p], j
    with pytest.raises(z.ZkbError, match="stride too small"):
        b.read_captured(0, n_batch, eb)   # a raw value does not fit an element's bytes
    b.close()


def test_gpu_capture_prime_call_group_outputs(monkeypatch):
    from tests.test_arith_call_groups_host import BLS12_381_FR, build, record
    monkeypatch.setenv("ZKB_TILE_LOG2", "3")
    r = build(BLS12_381_FR, 70, failing=True, n_asserts=1)
    n_batch = 50
    ws = [r.witness() for _ in range(n_batch)]
    W = np.array([[list(r.le(x % (1 << (8 * r.nb)))) for x in w] for w in ws], dtype=np.uint8)
    b, e = record(0, r.messages(r.witness()))
    assert b.stats()["n_call_groups"] >= 1
    assert e.get_violations() is not None   # the Evaluator's own finalize and one-witness run
    wires = [x for first, count in r.blocks for x in range(first, first + count, 5)]
    e.capture_wires(wires)
    v = b.evaluate(None, W, n_batch)
    handles = [e.value_handle(x) for x in wires]
    cap = check_against_read_values(b, handles, n_batch, 32)
    for j in (0, n_batch - 1):
        msgs = r.messages(ws[j])
        if ev.evaluate(msgs) == [] and v[j]["ok"]:
            o = ev.Evaluator.from_messages(msgs, ev.PlaintextBackend())
            assert as_ints(cap[j]) == [o.values[x] for x in wires], j


def test_gpu_capture_boolean_call_group_outputs():
    from tests.test_call_groups import build, record
    r = build(7, failing=True)
    b, e = record(0, r.messages(r.witness()))
    b.finalize(True)
    n_batch = 100
    rng = np.random.default_rng(3)
    W = rng.integers(0, 2, size=(n_batch, r.n_wit, 1)).astype(np.uint8)
    o0 = ev.Evaluator.from_messages(r.messages(W[0, :, 0]), ev.PlaintextBackend())
    wires = sorted(o0.values)
    handles = [e.value_handle(x) for x in wires]
    assert any(h >= 0x80000000 for h in handles)   # group outputs
    b.capture(handles)
    v = b.evaluate(None, W, n_batch)
    cap = check_against_read_values(b, handles, n_batch, 4)
    for j in (0, n_batch - 1):
        msgs = r.messages(W[j, :, 0])
        if ev.evaluate(msgs) == []:
            o = ev.Evaluator.from_messages(msgs, ev.PlaintextBackend())
            assert bool(v[j]["ok"])
            assert as_ints(cap[j]) == [o.values[x] for x in wires], j


def test_gpu_capture_two_contexts_on_one_device(monkeypatch):
    """zkb_evaluate_sharded over two contexts of device 0: each rank captures its block; concatenated, one context's capture"""
    monkeypatch.setenv("ZKB_TILE_LOG2", "5")
    c = circuits()
    z = zkb()
    p = FIELDS["bls381"]
    circ = c.random_circuit(1 << 12, 32, p, seed=2, n_tracked=8)
    n_batch = 301
    wit = c.make_witnesses(circ, n_batch, seed=3, corrupt={7: 1})
    one = z.GpuBackend(0)
    one.set_field(p)
    one.push_gates(circ.gates, circ.const_pool)
    one.finalize()
    handles = [h for _, h in live_wires(one, circ.n_wires)]
    one.capture(handles)
    v_one = one.evaluate(None, wit, n_batch)
    sh = z.ShardedBackend([0, 0])
    sh.root.set_field(p)
    sh.root.push_gates(circ.gates, circ.const_pool)
    sh.root.finalize()
    sh.capture(handles)   # broadcasts the program to the other rank first
    v = sh.evaluate(None, wit, n_batch)
    assert np.array_equal(v, v_one)
    assert np.array_equal(sh.read_captured(32), one.read_captured(0, n_batch, 32))
    v = sh.run()
    assert np.array_equal(sh.read_captured(32), one.read_captured(0, n_batch, 32))
    sh.close()
    one.close()


def test_gpu_capture_cpp_mirror(tmp_path):
    src = os.path.join(ROOT, "tests", "native", "capture_api.cpp")
    pkg = os.path.join(ROOT, "zkinterface-ir_b200")
    exe = str(tmp_path / "capture_api")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", exe, "-L", pkg, "-lzkb",
                           f"-Wl,-rpath,{pkg}"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == "capture_api ok"
