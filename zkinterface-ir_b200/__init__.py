"""zkb — B200-native satisfiability evaluator for the zkInterface SIEVE IR.

Host-side mirror of the reference's evaluation interface, over the C ABI of
`libzkb.so` (include/zkb.h):

  GpuBackend   `trait ZKBackend` (rust/src/consumers/evaluator.rs:17-76): same
               method names and argument meaning; deferred (records SSA ops),
               evaluated for a whole batch of witnesses by `evaluate`.
  Evaluator    `Evaluator<B>` (evaluator.rs:158-753): from_messages /
               ingest_message / get_violations / get, driven from `.sieve` bytes.
  Source       `Source` (rust/src/consumers/source.rs:59-118).

There is NO CPU fallback: without the CUDA library this module fails to import,
and without a GPU every evaluation call raises `ZkbError`.

The directory name contains a hyphen, so import it through `zkb_loader.load()`
(repo root) or `importlib`; it registers itself as module `zkir_b200`.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Iterable, List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ZKB_LIB_PATH") or os.path.join(_HERE, "libzkb.so")  # ZKB_LIB_PATH: a sanitized build (scripts/asan_host.sh)

if not os.path.exists(LIB_PATH):
    raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no CPU fallback)")
_lib = C.CDLL(LIB_PATH)

ZKB_OK, ZKB_E_ARG, ZKB_E_FORMAT, ZKB_E_SEMANTIC, ZKB_E_CUDA, ZKB_E_FATAL, ZKB_E_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
UINT64_MAX = (1 << 64) - 1

# zkb_gate_op
(G_CONSTANT, G_ASSERT_ZERO, G_COPY, G_ADD, G_MUL, G_ADD_CONSTANT, G_MUL_CONSTANT, G_AND, G_XOR, G_NOT, G_INSTANCE,
 G_WITNESS, G_FREE) = range(1, 14)

GATE_DTYPE = np.dtype([("op", "u1"), ("pad", "u1", (3,)), ("out", "<u4"), ("a", "<u4"), ("b", "<u4")])
VERDICT_DTYPE = np.dtype([("ok", "u1"), ("pad", "u1", (7,)), ("first_fail_seq", "<u8")])


class ZkbStats(C.Structure):
    _fields_ = [("n_values", C.c_uint64), ("n_asserts", C.c_uint64), ("n_instance", C.c_uint64),
                ("n_witness", C.c_uint64), ("n_consts", C.c_uint64), ("ir_gates", C.c_uint64),
                ("callbacks", C.c_uint64 * 12), ("n_slots", C.c_uint64), ("n_levels", C.c_uint64),
                ("n_device_ops", C.c_uint64), ("algo_bytes_per_witness", C.c_uint64), ("nlimb", C.c_uint32),
                ("binary", C.c_uint32), ("tile_witnesses", C.c_uint32), ("n_tiles", C.c_uint32),
                ("n_call_groups", C.c_uint64), ("n_group_calls", C.c_uint64),
                ("n_group_launches", C.c_uint64), ("n_group_table_slots", C.c_uint64), ("group_jit_state", C.c_int64),
                ("n_sink_ops", C.c_uint64), ("n_carried_groups", C.c_uint64)]


class ZkbTiming(C.Structure):
    _fields_ = [("h2d_ms", C.c_float), ("load_ms", C.c_float), ("levels_ms", C.c_float), ("total_ms", C.c_float),
                ("level_launches", C.c_uint64), ("kernel_launches", C.c_uint64)]


class ZkbCsr(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("row_ptr", C.c_void_p), ("col", C.c_void_p), ("coef_idx", C.c_void_p)]


CALLBACK_NAMES = ["constant", "instance", "witness", "add", "mul", "addc", "mulc", "and", "xor", "not", "copy",
                  "assert_zero"]

# every symbol include/zkb.h declares (tests check the library exports all of them)
EXPORTED = [
    "zkb_create", "zkb_destroy", "zkb_last_error", "zkb_set_limits", "zkb_set_field", "zkb_one", "zkb_minus_one", "zkb_zero", "zkb_copy",
    "zkb_constant", "zkb_assert_zero", "zkb_add", "zkb_multiply", "zkb_add_constant", "zkb_mul_constant", "zkb_and",
    "zkb_xor", "zkb_not", "zkb_instance", "zkb_witness", "zkb_push_gates", "zkb_finalize", "zkb_evaluate",
    "zkb_upload_inputs", "zkb_run", "zkb_assert_info", "zkb_pending_error", "zkb_read_values", "zkb_capture_values",
    "zkb_read_captured", "zkb_scope_lookup",
    "zkb_get_stats", "zkb_get_timing", "zkb_get_program", "zkb_get_const", "zkb_assert_value", "zkb_level_info", "zkb_evaluator_create", "zkb_evaluator_destroy", "zkb_evaluator_ingest_message",
    "zkb_evaluator_ingest_buffer", "zkb_evaluator_ingest_paths", "zkb_evaluator_get_violations",
    "zkb_evaluator_violation", "zkb_evaluator_get_wire", "zkb_evaluator_lookup", "zkb_evaluator_last_error", "zkb_evaluator_set_flatten", "zkb_evaluator_set_expand_definable", "zkb_evaluator_flatten",
    "zkb_evaluator_flatten_to_dir", "zkb_evaluator_add_value_set_buffer", "zkb_evaluator_add_value_set_paths",
    "zkb_evaluator_value_sets", "zkb_evaluator_use_devices", "zkb_evaluator_batch_result", "zkb_evaluator_batch_violation",
    "zkb_evaluator_get_wire_of", "zkb_debug_value_set_cut", "zkb_validator_create", "zkb_validator_destroy", "zkb_validator_ingest_message",
    "zkb_validator_ingest_buffer", "zkb_validator_ingest_paths", "zkb_validator_get_violations", "zkb_validator_violation",
    "zkb_validator_how_many_violations", "zkb_validator_live_wires", "zkb_validator_set_limits", "zkb_validator_last_error", "zkb_metrics_create", "zkb_metrics_destroy", "zkb_metrics_ingest_message",
    "zkb_metrics_ingest_buffer", "zkb_metrics_ingest_paths", "zkb_metrics_json", "zkb_metrics_last_error", "zkb_r1cs_load", "zkb_r1cs_check",
    "zkb_r1cs_upload", "zkb_r1cs_run", "zkb_debug_field_ops", "zkb_debug_field_throughput", "zkb_debug_group_jit_wait", "zkb_debug_group_jit_source", "zkb_debug_gather_throughput", "zkb_debug_barrier_cost", "zkb_debug_r1cs_layout", "zkb_debug_rewrite_message", "zkb_debug_plan_hash", "zkb_debug_plan_ops", "zkb_debug_write_flat_relation",
    "zkb_comm_unique_id", "zkb_comm_init_rank", "zkb_comm_init", "zkb_comm_info", "zkb_comm_broadcast_program", "zkb_comm_evaluate",
    "zkb_comm_run", "zkb_evaluate_sharded", "zkb_run_sharded",
]

_vp, _u8p, _sz, _u64, _u32, _i = C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_int
_u64p = C.POINTER(C.c_uint64)


def _sig(name, restype, *argtypes):
    f = getattr(_lib, name)
    f.restype = restype
    f.argtypes = list(argtypes)
    return f


_sig("zkb_create", _vp, _i)
_sig("zkb_destroy", None, _vp)
_sig("zkb_last_error", C.c_char_p, _vp)
_sig("zkb_pending_error", C.c_char_p, _vp)
_sig("zkb_set_limits", _i, _vp, _u64, _u64)
_sig("zkb_set_field", _i, _vp, _u8p, _sz, _u32, _i)
for _n in ("zkb_one", "zkb_minus_one", "zkb_zero"):
    _sig(_n, _i, _vp, _u8p, _sz, C.POINTER(C.c_size_t))
_sig("zkb_copy", _i, _vp, _u64, _u64p)
_sig("zkb_constant", _i, _vp, _u8p, _sz, _u64p)
_sig("zkb_assert_zero", _i, _vp, _u64, _u64)
for _n in ("zkb_add", "zkb_multiply", "zkb_and", "zkb_xor"):
    _sig(_n, _i, _vp, _u64, _u64, _u64p)
for _n in ("zkb_add_constant", "zkb_mul_constant"):
    _sig(_n, _i, _vp, _u64, _u8p, _sz, _u64p)
_sig("zkb_not", _i, _vp, _u64, _u64p)
_sig("zkb_instance", _i, _vp, _u64p)
_sig("zkb_witness", _i, _vp, _u64p)
_sig("zkb_push_gates", _i, _vp, _vp, _u64, _u8p, _sz, _u64)
_sig("zkb_finalize", _i, _vp, _i)
_sig("zkb_evaluate", _i, _vp, _u8p, _u64, _u8p, _u64, _u32, _u32, _vp)
_sig("zkb_upload_inputs", _i, _vp, _u8p, _u64, _u8p, _u64, _u32, _u32)
_sig("zkb_run", _i, _vp, _vp)
_sig("zkb_assert_info", _i, _vp, _u64, _u64p)
_sig("zkb_read_values", _i, _vp, _u32, _vp, _u64, _u8p, _sz)
_sig("zkb_capture_values", _i, _vp, _vp, _u64)
_sig("zkb_read_captured", _i, _vp, _u32, _u32, _u8p, _sz)
_sig("zkb_scope_lookup", _i, _vp, _u64, _u64p)
_sig("zkb_get_stats", _i, _vp, C.POINTER(ZkbStats))
_sig("zkb_get_timing", _i, _vp, C.POINTER(ZkbTiming))
_sig("zkb_get_program", _i, _vp, _u64, _u64, _vp, _vp, _vp)
_sig("zkb_get_const", _i, _vp, _u64, _u8p, _sz, C.POINTER(C.c_size_t))
_sig("zkb_assert_value", _i, _vp, _u64, _u64p)
_sig("zkb_level_info", _i, _vp, _u64, _vp)
_sig("zkb_evaluator_create", _vp, _vp)
_sig("zkb_evaluator_destroy", None, _vp)
_sig("zkb_evaluator_ingest_message", _i, _vp, _u8p, _sz)
_sig("zkb_evaluator_ingest_buffer", _i, _vp, _u8p, _sz)
_sig("zkb_evaluator_ingest_paths", _i, _vp, C.POINTER(C.c_char_p), _sz)
_sig("zkb_evaluator_get_violations", _i, _vp, C.POINTER(C.c_size_t))
_sig("zkb_evaluator_violation", C.c_char_p, _vp, _sz)
_sig("zkb_evaluator_get_wire", _i, _vp, _u64, _u8p, _sz, C.POINTER(C.c_size_t))
_sig("zkb_evaluator_lookup", _i, _vp, _u64, _u64p)
_sig("zkb_evaluator_last_error", C.c_char_p, _vp)
_sig("zkb_evaluator_set_flatten", _i, _vp, _i)
_sig("zkb_evaluator_set_expand_definable", _i, _vp, C.c_char_p)
_sig("zkb_evaluator_flatten", _i, _vp, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_void_p),
     C.POINTER(C.c_size_t), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t))
_sig("zkb_evaluator_flatten_to_dir", _i, _vp, C.c_char_p)
_sig("zkb_evaluator_add_value_set_buffer", _i, _vp, _u8p, _sz)
_sig("zkb_evaluator_add_value_set_paths", _i, _vp, C.POINTER(C.c_char_p), _sz)
_sig("zkb_evaluator_value_sets", _sz, _vp)
_sig("zkb_evaluator_use_devices", _i, _vp, C.POINTER(C.c_void_p), _i)
_sig("zkb_evaluator_batch_result", _i, _vp, _u64, C.POINTER(C.c_int), C.POINTER(C.c_size_t))
_sig("zkb_evaluator_batch_violation", C.c_char_p, _vp, _u64, _sz)
_sig("zkb_evaluator_get_wire_of", _i, _vp, _u64, _u64, _u8p, _sz, C.POINTER(C.c_size_t))
_sig("zkb_debug_value_set_cut", _i, _vp, _u64, _u64p, C.POINTER(C.c_int))
_sig("zkb_validator_create", _vp, _i)
_sig("zkb_validator_destroy", None, _vp)
_sig("zkb_validator_ingest_message", _i, _vp, _u8p, _sz)
_sig("zkb_validator_ingest_buffer", _i, _vp, _u8p, _sz)
_sig("zkb_validator_ingest_paths", _i, _vp, C.POINTER(C.c_char_p), _sz)
_sig("zkb_validator_get_violations", _i, _vp, C.POINTER(C.c_size_t))
_sig("zkb_validator_violation", C.c_char_p, _vp, _sz)
_sig("zkb_validator_how_many_violations", C.c_size_t, _vp)
_sig("zkb_validator_live_wires", _u64, _vp)
_sig("zkb_validator_set_limits", _i, _vp, _u64)
_sig("zkb_validator_last_error", C.c_char_p, _vp)
_sig("zkb_metrics_create", _vp)
_sig("zkb_metrics_destroy", None, _vp)
_sig("zkb_metrics_ingest_message", _i, _vp, _u8p, _sz)
_sig("zkb_metrics_ingest_buffer", _i, _vp, _u8p, _sz)
_sig("zkb_metrics_ingest_paths", _i, _vp, C.POINTER(C.c_char_p), _sz)
_sig("zkb_metrics_json", C.c_char_p, _vp)
_sig("zkb_metrics_last_error", C.c_char_p, _vp)
_sig("zkb_r1cs_load", _i, _vp, C.POINTER(ZkbCsr), C.POINTER(ZkbCsr), C.POINTER(ZkbCsr), _u8p, _sz, _u64, _u64)
_sig("zkb_r1cs_check", _i, _vp, _u8p, _u64, _u32, _u32, _vp)
_sig("zkb_r1cs_upload", _i, _vp, _u8p, _u64, _u32, _u32)
_sig("zkb_r1cs_run", _i, _vp, _vp)
_sig("zkb_debug_field_ops", _i, _vp, _i, _vp, _vp, _vp, _u64)
_sig("zkb_debug_field_throughput", _i, _vp, _i, _u32, C.POINTER(C.c_double))
_sig("zkb_debug_group_jit_wait", _i, _vp, C.POINTER(C.c_int), C.POINTER(C.c_double))
_sig("zkb_debug_group_jit_source", C.c_char_p, _vp)
_sig("zkb_debug_gather_throughput", _i, _vp, _u64, _u32, C.POINTER(C.c_double))
_sig("zkb_debug_barrier_cost", _i, _vp, _i, _u32, _u32, C.POINTER(C.c_double))
_sig("zkb_debug_r1cs_layout", _i, _vp, _i, _u64p, _vp, _vp, _vp)
_sig("zkb_debug_plan_hash", _i, _vp, _u64p)
_sig("zkb_debug_plan_ops", _i, _vp, _u64, _u64, _vp, _vp)
_sig("zkb_debug_rewrite_message", _i, _vp, _u8p, _sz, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t))
_sig("zkb_debug_write_flat_relation", _i, _vp, _u8p, _sz, _i, _vp, _u64, _u8p, _sz, _u64, C.POINTER(C.c_void_p),
     C.POINTER(C.c_size_t))
_sig("zkb_comm_unique_id", _i, _vp)
_sig("zkb_comm_init_rank", _i, _vp, _vp, _i, _i)
_sig("zkb_comm_init", _i, C.POINTER(C.c_void_p), _i)
_sig("zkb_comm_info", _i, _vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int))
_sig("zkb_comm_broadcast_program", _i, _vp, _i)
_sig("zkb_comm_evaluate", _i, _vp, _u8p, _u64, _u8p, _u64, _u32, _u32, _u32, _u32, _vp)
_sig("zkb_comm_run", _i, _vp, _u32, _u32, _vp)
_sig("zkb_evaluate_sharded", _i, C.POINTER(C.c_void_p), _i, _u8p, _u64, _u8p, _u64, _u32, _u32, _vp)
_sig("zkb_run_sharded", _i, C.POINTER(C.c_void_p), _i, _u32, _vp)


class ZkbError(Exception):
    """Non-zero zkb_status; `.code` is the status, str() the library's message
    (the reference's own error text where the reference has one)."""

    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


def _buf(b) -> C.c_void_p:
    """pointer to the bytes of a bytes / bytearray / numpy array (kept alive by the caller)"""
    if b is None:
        return None
    if isinstance(b, np.ndarray):
        return b.ctypes.data_as(C.c_void_p)
    if isinstance(b, bytes):
        return C.cast(C.c_char_p(b), C.c_void_p)  # points into `b`, which the caller keeps alive
    if isinstance(b, bytearray):
        return C.cast((C.c_char * len(b)).from_buffer(b), C.c_void_p)
    raise TypeError(type(b))


def _le(v, n=None) -> bytes:
    if isinstance(v, (bytes, bytearray)):
        return bytes(v)
    v = int(v)
    if n is None:
        n = max(1, (v.bit_length() + 7) // 8)
    return v.to_bytes(n, "little")


class GpuBackend:
    """Deferred, batched `ZKBackend` (evaluator.rs:17-76).  `Wire` = int (SSA handle),
    `FieldElement` = little-endian bytes or int."""

    def __init__(self, device: int = 0):
        self._c = _lib.zkb_create(device)
        self.device = device
        err = _lib.zkb_last_error(self._c).decode("utf-8", "replace")
        if device >= 0 and err:
            _lib.zkb_destroy(self._c)
            self._c = None
            raise ZkbError(ZKB_E_CUDA, err)
        self._keep = []

    def close(self):
        if getattr(self, "_c", None):
            _lib.zkb_destroy(self._c)
            self._c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != ZKB_OK:
            raise ZkbError(rc, _lib.zkb_last_error(self._c).decode("utf-8", "replace"))

    # ---- ZKBackend methods -------------------------------------------------
    @staticmethod
    def from_bytes_le(val: bytes) -> bytes:
        return bytes(val)

    def set_limits(self, max_values: int = 0, max_steps: int = 0):
        """resource limits of the host pass (0 keeps the current value), zkb.h section 1"""
        self._chk(_lib.zkb_set_limits(self._c, max_values, max_steps))

    def set_field(self, modulus, degree: int = 1, is_boolean: bool = False):
        m = _le(modulus)
        self._chk(_lib.zkb_set_field(self._c, _buf(m), len(m), degree, int(is_boolean)))

    def _elem(self, fn) -> bytes:
        out = C.create_string_buffer(64)
        n = C.c_size_t()
        self._chk(fn(self._c, C.cast(out, C.c_void_p), 64, C.byref(n)))
        return out.raw[:n.value]

    def one(self):
        return self._elem(_lib.zkb_one)

    def minus_one(self):
        return self._elem(_lib.zkb_minus_one)

    def zero(self):
        return self._elem(_lib.zkb_zero)

    def _w1(self, fn, *args):
        out = C.c_uint64()
        self._chk(fn(self._c, *args, C.byref(out)))
        return out.value

    def copy(self, a):
        return self._w1(_lib.zkb_copy, a)

    def constant(self, val):
        v = _le(val)
        return self._w1(_lib.zkb_constant, _buf(v), len(v))

    def assert_zero(self, a, src_wire_id: int = 0):
        self._chk(_lib.zkb_assert_zero(self._c, a, src_wire_id))

    def add(self, a, b):
        return self._w1(_lib.zkb_add, a, b)

    def multiply(self, a, b):
        return self._w1(_lib.zkb_multiply, a, b)

    def add_constant(self, a, val):
        v = _le(val)
        return self._w1(_lib.zkb_add_constant, a, _buf(v), len(v))

    def mul_constant(self, a, val):
        v = _le(val)
        return self._w1(_lib.zkb_mul_constant, a, _buf(v), len(v))

    def and_(self, a, b):
        return self._w1(_lib.zkb_and, a, b)

    def xor(self, a, b):
        return self._w1(_lib.zkb_xor, a, b)

    def not_(self, a):
        return self._w1(_lib.zkb_not, a)

    def instance(self, val=None):
        return self._w1(_lib.zkb_instance)

    def witness(self, val=None):
        return self._w1(_lib.zkb_witness)

    # ---- bulk gates / evaluation --------------------------------------------
    def push_gates(self, gates: np.ndarray, const_pool: Optional[np.ndarray] = None):
        """gates: GATE_DTYPE array; const_pool: uint8 [n_consts, stride]"""
        gates = np.ascontiguousarray(gates, dtype=GATE_DTYPE)
        if const_pool is None:
            const_pool = np.zeros((0, 1), dtype=np.uint8)
        const_pool = np.ascontiguousarray(const_pool, dtype=np.uint8)
        self._chk(_lib.zkb_push_gates(self._c, _buf(gates), len(gates), _buf(const_pool), const_pool.shape[1],
                                      const_pool.shape[0]))

    def finalize(self, keep_all_values: bool = False, verdicts_only: bool = False):
        """keep_all_values: every value readable (no slot re-use); verdicts_only: nothing readable"""
        self._chk(_lib.zkb_finalize(self._c, 1 if keep_all_values else (2 if verdicts_only else 0)))

    @staticmethod
    def _pack_inputs(x):
        """[n_batch, n_vals, stride] or [n_vals, stride] (shared) uint8 -> (array, set_stride, stride)"""
        if x is None:
            return None, 0, 0
        x = np.ascontiguousarray(x, dtype=np.uint8)
        if x.ndim == 2:
            return x, 0, x.shape[1]
        return x, x.shape[1] * x.shape[2], x.shape[2]

    def _strides(self, instances, witnesses, n_batch):
        inst, iss, istr = self._pack_inputs(instances)
        wit, wss, wstr = self._pack_inputs(witnesses)
        stride = wstr or istr or 1
        if istr and wstr and istr != wstr:
            raise ValueError("instance and witness value strides differ")
        # the C side reads n_batch sets of n_instance / n_witness values through these pointers: the arrays must hold them
        st = self.stats()
        for x, need, short in ((inst, st["n_instance"], (ZKB_E_SEMANTIC, "Not enough instance to consume")),          # evaluator.rs:420-427
                               (wit, st["n_witness"], (ZKB_E_FATAL, "Missing witness value for PlaintextBackend"))):  # :944-946
            if x is None:
                continue
            if x.ndim == 3 and x.shape[0] < n_batch:
                raise ZkbError(ZKB_E_ARG, f"input array holds {x.shape[0]} value sets, n_batch is {n_batch}")
            if x.ndim not in (2, 3):
                raise ZkbError(ZKB_E_ARG, "inputs must be [n_values, stride] or [n_batch, n_values, stride] uint8 arrays")
            if x.shape[-2] < need:
                raise ZkbError(*short)
        return inst, iss, wit, wss, stride

    def evaluate(self, instances, witnesses, n_batch: int) -> np.ndarray:
        """End-to-end: host buffers in, verdicts out (VERDICT_DTYPE array)."""
        inst, iss, wit, wss, stride = self._strides(instances, witnesses, n_batch)
        out = np.zeros(n_batch, dtype=VERDICT_DTYPE)
        self._chk(_lib.zkb_evaluate(self._c, _buf(inst), iss, _buf(wit), wss, stride, n_batch, _buf(out)))
        self._n_batch = n_batch          # the inputs stay resident: run() re-evaluates them
        return out

    def upload_inputs(self, instances, witnesses, n_batch: int):
        inst, iss, wit, wss, stride = self._strides(instances, witnesses, n_batch)
        self._chk(_lib.zkb_upload_inputs(self._c, _buf(inst), iss, _buf(wit), wss, stride, n_batch))
        self._n_batch = n_batch

    def resident_batch(self, n_batch: int):
        """the library itself uploaded the inputs of a batch of n_batch (an Evaluator's value sets): run() and
        read_captured() use them"""
        self._n_batch = n_batch

    def run(self) -> np.ndarray:
        if not getattr(self, "_n_batch", 0):
            raise ZkbError(ZKB_E_ARG, "run() needs inputs: call upload_inputs() or evaluate() first")
        out = np.zeros(self._n_batch, dtype=VERDICT_DTYPE)
        self._chk(_lib.zkb_run(self._c, _buf(out)))
        return out

    def assert_wire(self, seq: int) -> int:
        out = C.c_uint64()
        self._chk(_lib.zkb_assert_info(self._c, seq, C.byref(out)))
        return out.value

    def pending_error(self) -> Optional[str]:
        e = _lib.zkb_pending_error(self._c)
        return e.decode("utf-8", "replace") if e else None

    def read_values(self, batch_idx: int, values: Sequence[int], stride: int = 32) -> List[int]:
        vals = np.ascontiguousarray(values, dtype=np.uint64)
        out = np.zeros((len(vals), stride), dtype=np.uint8)
        self._chk(_lib.zkb_read_values(self._c, batch_idx, _buf(vals), len(vals), _buf(out), stride))
        return [int.from_bytes(out[i].tobytes(), "little") for i in range(len(vals))]

    def capture(self, values: Sequence[int]):
        """values (handles) whose canonical values every following run writes out for every witness of the batch (read them
        with read_captured); an empty list clears it"""
        vals = np.ascontiguousarray(values, dtype=np.uint64)
        self._chk(_lib.zkb_capture_values(self._c, _buf(vals), len(vals)))
        self._n_capture = len(vals)

    def read_captured(self, first: int = 0, n: Optional[int] = None, stride: Optional[int] = None) -> np.ndarray:
        """what the last run captured for witnesses [first, first + n): uint8 [n, n_values, stride], little-endian, the bytes
        read_values returns (n: to the end of the batch, one witness after a run the Evaluator made itself; stride: the
        field's element bytes)"""
        if n is None:
            n = getattr(self, "_n_batch", 1) - first
        if stride is None:
            st = self.stats()
            stride = 4 if st["binary"] else 4 * st["nlimb"]
        out = np.zeros((n, getattr(self, "_n_capture", 0), stride), dtype=np.uint8)
        self._chk(_lib.zkb_read_captured(self._c, first, n, _buf(out), stride))
        return out

    def scope_lookup(self, wire: int) -> int:
        out = C.c_uint64()
        self._chk(_lib.zkb_scope_lookup(self._c, wire, C.byref(out)))
        return out.value

    def program(self):
        """(kinds u8[n], a u32[n], b u32[n]) of the recorded SSA values"""
        n = self.stats()["n_values"]
        k = np.zeros(n, dtype=np.uint8)
        a = np.zeros(n, dtype=np.uint32)
        b = np.zeros(n, dtype=np.uint32)
        self._chk(_lib.zkb_get_program(self._c, 0, n, _buf(k), _buf(a), _buf(b)))
        return k, a, b

    def const_value(self, idx: int) -> int:
        out = C.create_string_buffer(64)
        n = C.c_size_t()
        self._chk(_lib.zkb_get_const(self._c, idx, C.cast(out, C.c_void_p), 64, C.byref(n)))
        return int.from_bytes(out.raw[:n.value], "little")

    def level_info(self, level: int) -> dict:
        out = np.zeros(5, dtype=np.uint64)
        self._chk(_lib.zkb_level_info(self._c, level, _buf(out)))
        return dict(zip(["gates", "arith", "fused_asserts", "not_stored", "algo_bytes_per_witness"], (int(x) for x in out)))

    def assert_value(self, seq: int) -> int:
        out = C.c_uint64()
        self._chk(_lib.zkb_assert_value(self._c, seq, C.byref(out)))
        return out.value

    def stats(self) -> dict:
        s = ZkbStats()
        self._chk(_lib.zkb_get_stats(self._c, C.byref(s)))
        d = {k: getattr(s, k) for k, _ in ZkbStats._fields_ if k != "callbacks"}
        d["callbacks"] = {n: s.callbacks[i] for i, n in enumerate(CALLBACK_NAMES)}
        return d

    def timing(self) -> dict:
        t = ZkbTiming()
        self._chk(_lib.zkb_get_timing(self._c, C.byref(t)))
        return {k: getattr(t, k) for k, _ in ZkbTiming._fields_}

    # ---- multi-GPU: one context per process (zkb.h section 7) ---------------------
    def comm_init_rank(self, comm_id: bytes, n_ranks: int, rank: int):
        """COLLECTIVE: join the communicator rank 0 created with comm_unique_id()"""
        cid = bytes(comm_id)
        if len(cid) != 128:
            raise ZkbError(ZKB_E_ARG, "comm id must be the 128 bytes of comm_unique_id()")
        self._chk(_lib.zkb_comm_init_rank(self._c, _buf(cid), n_ranks, rank))

    def comm_info(self) -> dict:
        r, n, t, v = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self._chk(_lib.zkb_comm_info(self._c, C.byref(r), C.byref(n), C.byref(t), C.byref(v)))
        return {"rank": r.value, "n_ranks": n.value, "transport": {0: "single", 1: "nccl", 2: "in-process"}[t.value],
                "nccl_version": v.value}

    def comm_broadcast_program(self, root: int = 0):
        """COLLECTIVE: the root's finalized program -> this rank (device plan over NCCL, no re-levelization)"""
        self._chk(_lib.zkb_comm_broadcast_program(self._c, root))

    def comm_evaluate(self, instances, witnesses, n_local: int, first: int, n_total: int) -> np.ndarray:
        """COLLECTIVE: this rank's witnesses [first, first + n_local) of a batch of n_total; verdicts of the whole batch"""
        inst, iss, wit, wss, stride = self._strides(instances, witnesses, n_local)
        out = np.zeros(n_total, dtype=VERDICT_DTYPE)
        self._chk(_lib.zkb_comm_evaluate(self._c, _buf(inst), iss, _buf(wit), wss, stride, n_local, first, n_total, _buf(out)))
        self._n_batch = n_local
        return out

    def comm_run(self, first: int, n_total: int) -> np.ndarray:
        """COLLECTIVE: the same over the resident inputs"""
        out = np.zeros(n_total, dtype=VERDICT_DTYPE)
        self._chk(_lib.zkb_comm_run(self._c, first, n_total, _buf(out)))
        return out

    # ---- debug / measurement ---------------------------------------------------
    def debug_field_ops(self, op: int, a: np.ndarray, b: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint32)
        b = np.ascontiguousarray(b, dtype=np.uint32)
        r = np.zeros_like(a)
        self._chk(_lib.zkb_debug_field_ops(self._c, op, _buf(a), _buf(b), _buf(r), a.shape[0]))
        return r

    def wait_group_jit(self):
        """block until the background compilation of the call groups' specialised kernel has ended -> (state, seconds):
        2 compiled (used from the next evaluation on), 3 loaded, -1 unavailable (the interpreter kernel stays), -2 no groups"""
        st, sec = C.c_int(), C.c_double()
        self._chk(_lib.zkb_debug_group_jit_wait(self._c, C.byref(st), C.byref(sec)))
        return st.value, sec.value

    def group_jit_source(self) -> str:
        return (_lib.zkb_debug_group_jit_source(self._c) or b"").decode()

    def debug_field_throughput(self, op: int, iters: int = 2000) -> float:
        out = C.c_double()
        self._chk(_lib.zkb_debug_field_throughput(self._c, op, iters, C.byref(out)))
        return out.value

    def debug_gather_throughput(self, table_bytes: int, iters: int = 64) -> float:
        """bytes / s of random 32-byte gathers from a table of table_bytes (the R1CS check's ceiling)"""
        out = C.c_double()
        self._chk(_lib.zkb_debug_gather_throughput(self._c, table_bytes, iters, C.byref(out)))
        return out.value

    def debug_barrier_cost(self, kind: int, blocks: int = 0, n_barriers: int = 200) -> float:
        """microseconds per barrier (0: cooperative_groups grid.sync, 1: the counter barrier of the all-levels kernel,
        2: one 8-CTA cluster's hardware barrier) with `blocks` CTAs (0: one per SM)"""
        out = C.c_double()
        self._chk(_lib.zkb_debug_barrier_cost(self._c, kind, blocks, n_barriers, C.byref(out)))
        return out.value

    # ---- R1CS -----------------------------------------------------------------
    def r1cs_load(self, A, B, Cm, coef_table: np.ndarray, n_vars: int):
        """A, B, Cm: (row_ptr uint64[n_rows+1], col uint32[nnz], coef_idx uint32[nnz])"""
        keep = []

        def mk(m):
            rp = np.ascontiguousarray(m[0], dtype=np.uint64)
            col = np.ascontiguousarray(m[1], dtype=np.uint32)
            ci = np.ascontiguousarray(m[2], dtype=np.uint32)
            keep.extend([rp, col, ci])
            return ZkbCsr(len(rp) - 1, rp.ctypes.data, col.ctypes.data, ci.ctypes.data)

        a, b, c = mk(A), mk(B), mk(Cm)
        coef_table = np.ascontiguousarray(coef_table, dtype=np.uint8)
        self._chk(_lib.zkb_r1cs_load(self._c, C.byref(a), C.byref(b), C.byref(c), _buf(coef_table),
                                     coef_table.shape[1], coef_table.shape[0], n_vars))

    def write_flat_relation(self, modulus: int, gates: np.ndarray, const_pool: Optional[np.ndarray] = None,
                            is_boolean: bool = False) -> bytes:
        """zkb_gate[] -> SIMPLE relation messages (100 000 gates each), as a GateBuilder over a MemorySink would emit"""
        gates = np.ascontiguousarray(gates)
        pool = np.ascontiguousarray(const_pool, dtype=np.uint8) if const_pool is not None else np.zeros((0, 1), np.uint8)
        m = _le(modulus)
        ptr, n = C.c_void_p(), C.c_size_t()
        self._chk(_lib.zkb_debug_write_flat_relation(self._c, _buf(m), len(m), int(is_boolean), gates.ctypes.data, len(gates),
                                                     _buf(pool), pool.shape[1], pool.shape[0], C.byref(ptr), C.byref(n)))
        return C.string_at(ptr.value, n.value)

    def plan_hash(self) -> int:
        out = C.c_uint64()
        self._chk(_lib.zkb_debug_plan_hash(self._c, C.byref(out)))
        return out.value

    def plan_ops(self, first: int = 0, n: int = -1, values: bool = False):
        """device ops [first, first + n) as uint32 [n, 4] {a, b, out, meta}; with values=True also the SSA value each op
        computes (0xFFFFFFFF: not stored; needs finalize(keep_all_values=True))"""
        if n < 0:
            n = self.stats()["n_device_ops"] - first
        ops = np.zeros((n, 4), dtype=np.uint32)
        vals = np.zeros(n, dtype=np.uint32) if values else None
        self._chk(_lib.zkb_debug_plan_ops(self._c, first, n, ops.ctypes.data, vals.ctypes.data if values else None))
        return (ops, vals) if values else ops

    def rewrite_message(self, buf: bytes) -> bytes:
        """C++ reader -> owned structs -> C++ writer (round-trip tests)"""
        ptr, n = C.c_void_p(), C.c_size_t()
        self._chk(_lib.zkb_debug_rewrite_message(self._c, _buf(buf), len(buf), C.byref(ptr), C.byref(n)))
        return C.string_at(ptr.value, n.value)

    def r1cs_layout(self, kind: int = 0):
        """(slices uint32[n,4], terms uint32[groups,32,2], row_ids uint32[rows]) of a host-only context"""
        cnt = (C.c_uint64 * 3)()
        self._chk(_lib.zkb_debug_r1cs_layout(self._c, kind, cnt, None, None, None))
        slices = np.zeros((cnt[0], 4), dtype=np.uint32)
        terms = np.zeros((cnt[1], 32, 2), dtype=np.uint32)
        rows = np.zeros(cnt[2], dtype=np.uint32)
        self._chk(_lib.zkb_debug_r1cs_layout(self._c, kind, cnt, slices.ctypes.data, terms.ctypes.data, rows.ctypes.data))
        return slices, terms, rows

    def r1cs_check(self, z: np.ndarray) -> np.ndarray:
        """z: uint8 [n_batch, n_vars, stride]"""
        z = np.ascontiguousarray(z, dtype=np.uint8)
        out = np.zeros(z.shape[0], dtype=VERDICT_DTYPE)
        self._chk(_lib.zkb_r1cs_check(self._c, _buf(z), z.shape[1] * z.shape[2], z.shape[2], z.shape[0], _buf(out)))
        return out

    def r1cs_upload(self, z: np.ndarray):
        z = np.ascontiguousarray(z, dtype=np.uint8)
        self._chk(_lib.zkb_r1cs_upload(self._c, _buf(z), z.shape[1] * z.shape[2], z.shape[2], z.shape[0]))
        self._n_batch = z.shape[0]

    def r1cs_run(self) -> np.ndarray:
        out = np.zeros(self._n_batch, dtype=VERDICT_DTYPE)
        self._chk(_lib.zkb_r1cs_run(self._c, _buf(out)))
        return out


def comm_unique_id() -> bytes:
    """rank 0 of a one-process-per-GPU job: the id every rank passes to GpuBackend.comm_init_rank (zkb.h section 7)"""
    out = C.create_string_buffer(128)
    rc = _lib.zkb_comm_unique_id(C.cast(out, C.c_void_p))
    if rc != ZKB_OK:
        raise ZkbError(rc, "zkb_comm_unique_id failed (NCCL not available?)")
    return out.raw


class ShardedBackend:
    """One process, N devices (zkb.h section 7): `backends[0]` records and finalizes the relation, the others receive its
    device plan on first use; a batch is split into N contiguous blocks, the verdicts MIN-reduced over NCCL."""

    def __init__(self, devices: Sequence[int]):
        self.backends = [GpuBackend(d) for d in devices]
        self._arr = (C.c_void_p * len(self.backends))(*[b._c for b in self.backends])
        rc = _lib.zkb_comm_init(self._arr, len(self.backends))
        if rc != ZKB_OK:
            msg = _lib.zkb_last_error(self.backends[0]._c).decode("utf-8", "replace")
            self.close()
            raise ZkbError(rc, msg)
        self.root = self.backends[0]
        self._n_batch = 0
        self._replicated = False  # the other ranks hold the root's program (the root finalizes once)

    def close(self):
        for b in getattr(self, "backends", []):
            b.close()

    def shard_of(self, rank: int, n_batch: int):
        n = len(self.backends)
        return n_batch * rank // n, n_batch * (rank + 1) // n

    def owner(self, j: int, n_batch: int):
        """(backend holding witness j, its index there)"""
        for r, b in enumerate(self.backends):
            lo, hi = self.shard_of(r, n_batch)
            if lo <= j < hi:
                return b, j - lo
        raise IndexError(j)

    def evaluate(self, instances, witnesses, n_batch: int) -> np.ndarray:
        inst, iss, wit, wss, stride = self.root._strides(instances, witnesses, n_batch)
        out = np.zeros(n_batch, dtype=VERDICT_DTYPE)
        self.root._chk(_lib.zkb_evaluate_sharded(self._arr, len(self.backends), _buf(inst), iss, _buf(wit), wss, stride, n_batch,
                                                 _buf(out)))
        self._n_batch = n_batch
        self._replicated = True
        return out

    def resident_batch(self, n_batch: int):
        """the library itself evaluated a batch of n_batch over these contexts (zkb_evaluate_sharded, e.g. an Evaluator's
        value sets): every rank holds the program and its block of the inputs; run() and read_captured() use them"""
        self._n_batch = n_batch
        self._replicated = True

    def run(self) -> np.ndarray:
        out = np.zeros(self._n_batch, dtype=VERDICT_DTYPE)
        self.root._chk(_lib.zkb_run_sharded(self._arr, len(self.backends), self._n_batch, _buf(out)))
        return out

    def _fan_out(self, fn):
        """fn(backend) on every rank at once (a collective blocks until every rank has joined it)"""
        errs = [None] * len(self.backends)

        def one(i):
            try:
                fn(self.backends[i])
            except ZkbError as e:
                errs[i] = e

        th = [threading.Thread(target=one, args=(i,)) for i in range(1, len(self.backends))]
        for t in th:
            t.start()
        one(0)
        for t in th:
            t.join()
        for e in errs:
            if e is not None:
                raise e

    def capture(self, values: Sequence[int]):
        """the same capture list on every rank (handles of the root's program); the ranks that have not received the
        program yet get it first"""
        if len(self.backends) > 1 and not self._replicated:
            self._fan_out(lambda b: b.comm_broadcast_program(0))
            self._replicated = True
        for b in self.backends:
            b.capture(values)

    def read_captured(self, stride: Optional[int] = None) -> np.ndarray:
        """what the last run captured for the whole batch, in batch order: uint8 [n_batch, n_values, stride]"""
        return np.concatenate([b.read_captured(0, hi - lo, stride)
                               for b, (lo, hi) in zip(self.backends, (self.shard_of(r, self._n_batch) for r in range(len(self.backends))))])


class Source:
    """`Source` (rust/src/consumers/source.rs:45-118): where `.sieve` messages come from."""

    def __init__(self, paths=None, buffers=None):
        self.paths = paths
        self.buffers = buffers

    @classmethod
    def from_directory(cls, path):
        return cls(paths=[str(path)])

    @classmethod
    def from_dirs_and_files(cls, paths):
        return cls(paths=[str(p) for p in paths])

    @classmethod
    def from_buffers(cls, buffers: Iterable[bytes]):
        return cls(buffers=[bytes(b) for b in buffers])


class Evaluator:
    """`Evaluator<GpuBackend>` (evaluator.rs:158-753) over `.sieve` bytes."""

    def __init__(self, backend: Optional[GpuBackend] = None, device: int = 0, flatten: bool = False,
                 expand_gate_set: Optional[str] = None):
        """flatten=True: the Evaluator drives the IRFlattener instead of an evaluating backend
        (consumers/flattening.rs); the statement can then be written out with flatten() / flatten_to_dir()."""
        flatten = flatten or expand_gate_set is not None
        self.backend = backend or GpuBackend(-1 if flatten else device)
        self._e = _lib.zkb_evaluator_create(self.backend._c)
        self._n_sets = 0
        self._sharded = None
        if expand_gate_set is not None:   # ExpandDefinable in front of the flattener (consumers/exp_definable.rs)
            self._chk(_lib.zkb_evaluator_set_expand_definable(self._e, expand_gate_set.encode()))
        elif flatten:
            self._chk(_lib.zkb_evaluator_set_flatten(self._e, 1))

    def close(self):
        if getattr(self, "_e", None):
            _lib.zkb_evaluator_destroy(self._e)
            self._e = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != ZKB_OK:
            raise ZkbError(rc, _lib.zkb_evaluator_last_error(self._e).decode("utf-8", "replace"))

    @classmethod
    def from_messages(cls, source: Source, backend: Optional[GpuBackend] = None, device: int = 0):
        ev = cls(backend, device)
        ev.ingest_source(source)
        return ev

    def ingest_source(self, source: Source):
        if source.buffers is not None:
            for b in source.buffers:
                self._chk(_lib.zkb_evaluator_ingest_buffer(self._e, _buf(b), len(b)))
        else:
            arr = (C.c_char_p * len(source.paths))(*[p.encode() for p in source.paths])
            self._chk(_lib.zkb_evaluator_ingest_paths(self._e, arr, len(source.paths)))

    def ingest_message(self, buf: bytes):
        self._chk(_lib.zkb_evaluator_ingest_message(self._e, _buf(buf), len(buf)))

    def get_violations(self) -> List[str]:
        n = C.c_size_t()
        self._chk(_lib.zkb_evaluator_get_violations(self._e, C.byref(n)))
        return [_lib.zkb_evaluator_violation(self._e, i).decode("utf-8", "replace") for i in range(n.value)]

    def flatten(self):
        """(instance, witness, relation) buffers of size-prefixed messages — IRFlattener over a MemorySink"""
        ptr = [C.c_void_p() for _ in range(3)]
        ln = [C.c_size_t() for _ in range(3)]
        self._chk(_lib.zkb_evaluator_flatten(self._e, C.byref(ptr[0]), C.byref(ln[0]), C.byref(ptr[1]), C.byref(ln[1]),
                                             C.byref(ptr[2]), C.byref(ln[2])))
        return tuple(C.string_at(p.value, n.value) if n.value else b"" for p, n in zip(ptr, ln))

    def flatten_to_dir(self, out_dir):
        """IRFlattener over FilesSink::new_clean: 000_instance / 001_witness / 002_relation .sieve"""
        self._chk(_lib.zkb_evaluator_flatten_to_dir(self._e, str(out_dir).encode()))

    def value_handle(self, wire_id: int) -> int:
        """SSA handle bound to a live top-scope wire (for GpuBackend.read_values on any batch element)"""
        out = C.c_uint64()
        self._chk(_lib.zkb_evaluator_lookup(self._e, wire_id, C.byref(out)))
        return out.value

    def capture_wires(self, wire_ids: Sequence[int]):
        """capture the live top-scope wires wire_ids on every following run of the backend (GpuBackend.capture); their
        values come back from backend.read_captured() in this order.  With value sets: a capture list can only be set on a
        finalized program, so the batch is evaluated (once, if get_batch_violations has not done it) and then run once more
        with the list; read_captured() of the backend that ran it (the ShardedBackend given to use_devices when the batch was
        split, else `backend`) returns [set, wire, bytes] for every set.  The values are those of the relation recorded in
        full: for a set whose recording stops early (value_set_cut(set)[0] != 0), values defined after its cut are computed
        from zero-padded inputs and are not part of its statement."""
        handles = [self.value_handle(w) for w in wire_ids]
        if not self._n_sets:
            self.backend.capture(handles)
            return
        self.get_batch_violations()
        runner = self._batch_runner()
        runner.resident_batch(self._n_sets)
        runner.capture(handles)
        runner.run()

    # ---- value sets: one relation, many instance / witness sets (zkb.h section 4) ----------------------------------
    def add_value_set(self, source: Source):
        """one value set (Instance / Witness messages); every set comes before the first relation message"""
        if source.buffers is not None:
            b = b"".join(source.buffers)
            self._chk(_lib.zkb_evaluator_add_value_set_buffer(self._e, _buf(b), len(b)))
        else:
            arr = (C.c_char_p * len(source.paths))(*[p.encode() for p in source.paths])
            self._chk(_lib.zkb_evaluator_add_value_set_paths(self._e, arr, len(source.paths)))
        self._n_sets = int(_lib.zkb_evaluator_value_sets(self._e))

    def use_devices(self, sharded: ShardedBackend):
        """split the batch over sharded's contexts; sharded.root must be this evaluator's backend"""
        self._chk(_lib.zkb_evaluator_use_devices(self._e, sharded._arr, len(sharded.backends)))
        self._sharded = sharded

    def get_batch_violations(self) -> List[tuple]:
        """[(status, violations)] per set: (ZKB_OK, what get_violations returns for the set's statement) or
        (ZKB_E_FATAL, [panic text]) where that statement makes the reference panic"""
        out = []
        st, n = C.c_int(), C.c_size_t()
        for j in range(self._n_sets):
            self._chk(_lib.zkb_evaluator_batch_result(self._e, j, C.byref(st), C.byref(n)))
            out.append((st.value, [_lib.zkb_evaluator_batch_violation(self._e, j, i).decode("utf-8", "replace")
                                   for i in range(n.value)]))
        if not self._n_sets:   # the library's refusal
            self._chk(_lib.zkb_evaluator_batch_result(self._e, 0, C.byref(st), C.byref(n)))
        return out

    def get_of(self, set_index: int, wire_id: int) -> int:
        """Evaluator.get for one value set (ZKB_E_ARG for a set whose recording stops early: value_set_cut)"""
        out = C.create_string_buffer(64)
        n = C.c_size_t()
        self._chk(_lib.zkb_evaluator_get_wire_of(self._e, set_index, wire_id, C.cast(out, C.c_void_p), 64, C.byref(n)))
        return int.from_bytes(out.raw[:n.value], "little")

    def value_set_cut(self, set_index: int):
        """(what, seq) of a set's cut point, from the recording alone: what 0 none, 1 instance stream empty, 2 witness
        stream empty, 3 the recording's own error / panic; seq = assertions recorded before it (None: no cut)"""
        seq, what = C.c_uint64(), C.c_int()
        self._chk(_lib.zkb_debug_value_set_cut(self._e, set_index, C.byref(seq), C.byref(what)))
        return what.value, (None if what.value == 0 else seq.value)

    def _batch_runner(self):
        sh = self._sharded
        return sh if sh is not None and len(sh.backends) > 1 and self._n_sets >= len(sh.backends) else self.backend

    def get(self, wire_id: int) -> int:
        out = C.create_string_buffer(64)
        n = C.c_size_t()
        self._chk(_lib.zkb_evaluator_get_wire(self._e, wire_id, C.cast(out, C.c_void_p), 64, C.byref(n)))
        return int.from_bytes(out.raw[:n.value], "little")


class Validator:
    """`Validator` (rust/src/consumers/validator.rs:68-829) over `.sieve` bytes; host only."""

    def __init__(self, as_prover: bool = False):
        self._v = _lib.zkb_validator_create(int(as_prover))

    @classmethod
    def new_as_prover(cls):
        return cls(True)

    @classmethod
    def new_as_verifier(cls):
        return cls(False)

    def close(self):
        if getattr(self, "_v", None):
            _lib.zkb_validator_destroy(self._v)
            self._v = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != ZKB_OK:
            raise ZkbError(rc, _lib.zkb_validator_last_error(self._v).decode("utf-8", "replace"))

    def set_limits(self, max_steps: int):
        self._chk(_lib.zkb_validator_set_limits(self._v, max_steps))

    def ingest_message(self, buf: bytes):
        self._chk(_lib.zkb_validator_ingest_message(self._v, _buf(buf), len(buf)))

    def ingest_source(self, source: Source):
        if source.buffers is not None:
            for b in source.buffers:
                self._chk(_lib.zkb_validator_ingest_buffer(self._v, _buf(b), len(b)))
        else:
            arr = (C.c_char_p * len(source.paths))(*[p.encode() for p in source.paths])
            self._chk(_lib.zkb_validator_ingest_paths(self._v, arr, len(source.paths)))

    def how_many_violations(self) -> int:
        return int(_lib.zkb_validator_how_many_violations(self._v))

    def live_wires(self) -> int:
        return int(_lib.zkb_validator_live_wires(self._v))

    def get_violations(self) -> List[str]:
        n = C.c_size_t()
        self._chk(_lib.zkb_validator_get_violations(self._v, C.byref(n)))
        return [_lib.zkb_validator_violation(self._v, i).decode("utf-8", "replace") for i in range(n.value)]


class Stats:
    """`Stats` (rust/src/consumers/stats.rs) over `.sieve` bytes; host only."""

    def __init__(self):
        self._m = _lib.zkb_metrics_create()

    def close(self):
        if getattr(self, "_m", None):
            _lib.zkb_metrics_destroy(self._m)
            self._m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != ZKB_OK:
            raise ZkbError(rc, _lib.zkb_metrics_last_error(self._m).decode("utf-8", "replace"))

    def ingest_message(self, buf: bytes):
        self._chk(_lib.zkb_metrics_ingest_message(self._m, _buf(buf), len(buf)))

    def ingest_source(self, source: Source):
        if source.buffers is not None:
            for b in source.buffers:
                self._chk(_lib.zkb_metrics_ingest_buffer(self._m, _buf(b), len(b)))
        else:
            arr = (C.c_char_p * len(source.paths))(*[p.encode() for p in source.paths])
            self._chk(_lib.zkb_metrics_ingest_paths(self._m, arr, len(source.paths)))

    def to_json_pretty(self) -> str:
        return _lib.zkb_metrics_json(self._m).decode("utf-8", "replace")
