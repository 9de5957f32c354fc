"""Capture list (zkb_capture_values / zkb_read_captured) on a host-only context: argument errors, clearing, the ZKB_E_CUDA of
every evaluation call, and a plan the list leaves unchanged."""
import ctypes as C

import numpy as np
import pytest

from tests.util import FIELDS, circuits, random_flat_program, zkb


def _backend(keep_values, p=FIELDS["bls381"]):
    z = zkb()
    gates, pool, _ = random_flat_program(p, 2000, 3, 5, seed=21)
    b = z.GpuBackend(-1)
    b.set_field(p)
    b.push_gates(gates, pool)
    if keep_values is not None:
        b.finalize(keep_all_values=keep_values == 1, verdicts_only=keep_values == 2)
    return z, b


def _capture_rc(z, b, handles):
    vals = np.ascontiguousarray(handles, dtype=np.uint64)
    rc = z._lib.zkb_capture_values(b._c, vals.ctypes.data_as(C.c_void_p), len(vals))
    return rc, z._lib.zkb_last_error(b._c).decode()


def _unreadable(b):
    """a gate value that is not stored under the current finalize (slot re-use / verdicts only)"""
    kinds, _, _ = b.program()
    for h in range(len(kinds) - 1, -1, -1):
        if kinds[h] > 2:   # not an input (inputs stay readable from their raw streams)
            try:
                b.capture([h])
            except zkb().ZkbError as e:
                return h, e
    raise AssertionError("every value is readable")


def test_capture_before_finalize_is_refused():
    z, b = _backend(None)
    rc, msg = _capture_rc(z, b, [0])
    assert rc == z.ZKB_E_ARG and "finalize" in msg
    b.close()


def test_unknown_handle_is_refused():
    z, b = _backend(1)
    n = b.stats()["n_values"]
    for h in (n, n + 5, 0x80000000, 2 ** 63):
        rc, msg = _capture_rc(z, b, [0, h])
        assert rc == z.ZKB_E_ARG and msg == "unknown wire handle", h
    b.close()


@pytest.mark.parametrize("keep_values", [0, 2])
def test_unreadable_value_is_refused(keep_values):
    z, b = _backend(keep_values)
    h, e = _unreadable(b)
    assert e.code == z.ZKB_E_ARG and "was not kept on device" in str(e)
    b.close()


def test_keep_all_accepts_every_value_and_n0_clears():
    z, b = _backend(1)
    n = b.stats()["n_values"]
    b.capture(list(range(n)))
    b.capture([])
    rc, _ = _capture_rc(z, b, [])
    assert rc == z.ZKB_OK
    b.close()


def test_read_captured_on_a_host_only_context_is_a_cuda_error():
    z, b = _backend(1)
    out = np.zeros(64, dtype=np.uint8)
    b.capture([0, 1])
    with pytest.raises(z.ZkbError) as e:
        b.read_captured(0, 1, 32)
    assert e.value.code == z.ZKB_E_CUDA
    b.close()
    z2, nb = _backend(None)
    rc = z2._lib.zkb_read_captured(nb._c, 0, 1, out.ctypes.data_as(C.c_void_p), 32)
    assert rc == z2.ZKB_E_ARG and "finalize" in z2._lib.zkb_last_error(nb._c).decode()
    nb.close()


def test_a_capture_list_leaves_the_plan_unchanged():
    c = circuits()
    z = zkb()
    circ = c.random_circuit(1 << 12, 32, FIELDS["bls381"], seed=6, n_tracked=8)
    b = z.GpuBackend(-1)
    b.set_field(FIELDS["bls381"])
    b.push_gates(circ.gates, circ.const_pool)
    b.finalize()
    h0, ops0 = b.plan_hash(), b.plan_ops()
    info0 = [b.level_info(l) for l in range(b.stats()["n_levels"])]
    live = [b.scope_lookup(w) for w in range(circ.n_wires) if _bound(b, w)]
    b.capture(live)
    assert b.plan_hash() == h0 and np.array_equal(b.plan_ops(), ops0)
    assert [b.level_info(l) for l in range(b.stats()["n_levels"])] == info0
    b.capture([])
    assert b.plan_hash() == h0
    b.close()


def _bound(b, w):
    try:
        b.scope_lookup(w)
        return True
    except zkb().ZkbError:
        return False
