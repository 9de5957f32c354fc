"""FieldParams::mul_form (Program::set_field): the hot kernels take the low-word Montgomery product exactly for 8-limb moduli
whose low 64 bits are 2^64 - 2^32 + 1."""
import ctypes as C

import pytest

from tests.test_field_host import lib  # noqa: F401  (fixture)
from tests.util import FIELDS

LOW = 0xFFFFFFFF00000001
FORM_WORD = 27  # FieldParams: p, r2, one (8 limbs each), n0inv, nlimb, top_mask, mul_form

CASES = {
    **{name: int(name == "bls381") for name in FIELDS},     # goldilocks has the low word but 2 limbs
    "top_ffffffff": ((0xFFFFFFFF << 224) | (0x1234 << 100) | LOW, 1),
    "just_above_2p224": ((1 << 224) | (0xABCDEF << 70) | LOW, 1),
    "random_high": ((0x5EED << 240) | (0x9E3779B97F4A7C15 << 128) | LOW, 1),
    "four_limbs": ((1 << 100) | LOW, 0),
    "low_word_off_by_2": ((1 << 255) | (LOW + 2), 0),
    "high_half_only": ((1 << 255) | (0xFFFFFFFF << 32) | 3, 0),
}


@pytest.mark.parametrize("name", list(CASES))
def test_mul_form_flag(lib, name):  # noqa: F811
    case = CASES[name]
    p, want = (FIELDS[name], case) if name in FIELDS else case
    fp = (C.c_uint32 * 28)()
    mod = p.to_bytes((p.bit_length() + 7) // 8, "little")
    n = lib.field_host_params(mod, len(mod), fp)
    assert fp[FORM_WORD] == want, (name, hex(p))
    if want:
        assert n == 8 and fp[24] == 0xFFFFFFFF  # n0inv = -1: the row multiplier is -T0
