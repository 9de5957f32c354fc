"""The Montgomery product for 8-limb moduli whose low 64 bits are 2^64 - 2^32 + 1 (field_ptx.cuh: fe_mont_mul_low64, the
hot kernels' product at BLS12-381 Fr) against Python integers and the portable CIOS product, bit for bit.  The product
needs no prime: odd moduli of that form with random high limbs, one near 2^256 (the top carry) and one just above 2^224,
and operands that make a row's bottom limb zero (m = 0)."""
import numpy as np
import pytest

from tests.test_field_host import limbs, unlimbs
from tests.test_gpu_flat import _check
from tests.util import FIELDS, circuits, random_flat_program, zkb

pytestmark = pytest.mark.gpu

LOW = 0xFFFFFFFF00000001


def _moduli():
    rng = np.random.default_rng(2024)
    mid = lambda k: int.from_bytes(rng.bytes(4 * k), "little")
    out = {"bls381": FIELDS["bls381"],
           "top_ffffffff": (0xFFFFFFFF << 224) | (mid(5) << 64) | LOW,
           "just_above_2p224": (1 << 224) | (mid(5) << 64) | LOW}
    for i in range(3):
        out[f"random{i}"] = (mid(6) << 64) | LOW | (1 << 255 - i)
    return out


MODULI = _moduli()


@pytest.mark.parametrize("name", list(MODULI))
def test_low64_product_matches_integers(name):
    z = zkb()
    p = MODULI[name]
    b = z.GpuBackend(0)
    b.set_field(p)
    assert b.stats()["nlimb"] == 8
    R = 1 << 256
    rng = np.random.default_rng(11)
    rand = lambda: int.from_bytes(rng.bytes(32), "little") % p
    # operands whose low limbs are zero keep a row's bottom limb T0 (and so m) zero for one or more rows
    zero_rows = [0, 1 << 32, 3 << 64, 5 << 96, 7 << 160, 1 << 224, (p - 1) >> 32 << 32, R % p]
    edge = [0, 1, 2, p - 1, p - 2, (p - 1) // 2, (p + 1) // 2, R % p, (R * R) % p] + [v % p for v in zero_rows]
    xs = edge + edge + [rand() for _ in range(20000)]
    ys = list(reversed(edge)) + [rand() for _ in edge] + [rand() for _ in range(20000)]
    A, B = limbs(xs, 8), limbs(ys, 8)
    Rinv = pow(R, -1, p)
    want = [x * y * Rinv % p for x, y in zip(xs, ys)]
    assert unlimbs(b.debug_field_ops(1, A, B)) == want      # the hot kernels' product for this form
    assert unlimbs(b.debug_field_ops(2, A, B)) == want      # portable CIOS
    # an unreduced first operand (any 8-limb integer) times a reduced one, as k_load_inputs does with R^2
    us = [R - 1, p, p + 1, R - (1 << 32)] + zero_rows + [int.from_bytes(rng.bytes(32), "little") for _ in range(5000)]
    r2 = [(R * R) % p] * len(us)
    assert unlimbs(b.debug_field_ops(1, limbs(us, 8), limbs(r2, 8))) == [u * R % p for u in us]
    b.close()


@pytest.mark.parametrize("name,tile_log2,tma", [("bls381", "8", "0"), ("bls381", "5", "1"), ("top_ffffffff", "8", "1"),
                                                ("top_ffffffff", "8", "0"), ("just_above_2p224", "8", "1"), ("just_above_2p224", "5", "1")])
def test_low64_level_path_parity(name, tile_log2, tma, monkeypatch):
    """One launch per wavefront (ZKB_COOP=0) with the low-word product, against the oracle: k_level_tma on 256-lane tiles,
    k_level_pipe on them with ZKB_LEVEL_TMA=0 and on narrow tiles"""
    monkeypatch.setenv("ZKB_COOP", "0")
    monkeypatch.setenv("ZKB_LEVEL_TMA", tma)
    monkeypatch.setenv("ZKB_TILE_LOG2", tile_log2)
    c = circuits()
    p = MODULI[name]
    n_batch = 256 + 45
    gates, pool, n_wires = random_flat_program(p, 900, 4, 6, seed=9, bool_ops=False)
    rng = np.random.default_rng(13)
    inst = c.random_field_elements(rng, (4,), p)
    wit = c.random_field_elements(rng, (n_batch, 6), p)
    _, _, st = _check(c, gates, pool, p, inst, wit, n_batch, n_wires, sample=(0, 255, n_batch - 1))
    assert st["tile_witnesses"] == 1 << int(tile_log2)
