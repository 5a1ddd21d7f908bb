"""CPU checks of the filtered stage-I search's host side: row tags and query masks become int32 bit patterns (0xFFFFFFFF <-> -1);
values outside [0, 2^32) and non-integers are rejected before anything reaches the device."""
import numpy as np
import pytest

import cir_b200 as cir

tag_bits = cir.engine.tag_bits


def test_python_ints_become_bit_patterns():
    assert tag_bits(0).dtype == np.int32 and int(tag_bits(0)) == 0
    assert int(tag_bits(5)) == 5
    assert int(tag_bits(0x7FFFFFFF)) == 0x7FFFFFFF
    assert int(tag_bits(0x80000000)) == -(1 << 31)
    assert int(tag_bits(0xFFFFFFFF)) == -1 == int(tag_bits(cir.engine.ALL_TAGS))
    assert tag_bits([1, 2, 4, 0xFFFFFFFF]).tolist() == [1, 2, 4, -1]


def test_numpy_arrays():
    u = np.array([0, 1, 0x80000001, 0xFFFFFFFF], dtype=np.uint32)
    b = tag_bits(u)
    assert b.dtype == np.int32 and np.array_equal(b.view(np.uint32), u)
    assert tag_bits(np.array([3, 0xFFFFFFFF], dtype=np.int64)).tolist() == [3, -1]
    assert tag_bits(np.array([7], dtype=np.uint64)).tolist() == [7]
    assert tag_bits(np.uint32(0xFFFFFFFE)).item() == -2
    assert tag_bits(np.zeros((0,), dtype=np.uint32)).shape == (0,)


@pytest.mark.parametrize("bad", [-1, 1 << 32, [1, -5], np.array([1 << 33], dtype=np.int64), np.array([-1], dtype=np.int32),
                                 np.array([1 << 63], dtype=np.uint64), 1 << 70])
def test_out_of_range_is_rejected(bad):
    with pytest.raises(ValueError, match=r"\[0, 2\^32\)"):
        tag_bits(bad)


@pytest.mark.parametrize("bad", [1.0, np.array([1.5]), True, np.array([True, False]), "3"])
def test_non_integers_are_rejected(bad):
    with pytest.raises(TypeError):
        tag_bits(bad)
