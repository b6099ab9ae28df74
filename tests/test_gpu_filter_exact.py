"""The EPF stages of the vector filter path take 1 / (sum of weights) with a reciprocal built from the approximate
hardware reciprocal and one FMA correction instead of the IEEE divide. The sum always lies in [1, 5]; this checks on the
device that the two agree bit for bit on every float of that range."""
import ctypes as C

import pytest

from jxl_rs_b200 import abi

pytestmark = pytest.mark.gpu


def test_epf_reciprocal_matches_ieee_divide_on_1_to_5():
    lib = abi.load_library()
    fn = lib.jxg_test_recip_1_5_mismatches
    fn.argtypes = [C.POINTER(C.c_ulonglong), C.POINTER(C.c_uint32)]
    fn.restype = C.c_int
    n, first = C.c_ulonglong(), C.c_uint32()
    assert fn(C.byref(n), C.byref(first)) == 0, "CUDA error in the reciprocal check"
    assert n.value == 0, f"{n.value} floats in [1, 5] differ from 1.0f / x, the first at bits 0x{first.value:08x}"
