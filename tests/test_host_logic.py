"""CPU-only checks of the host side: the C ABI library loads and exports every symbol the
header declares, descriptor layouts agree, the build refuses to pretend without a GPU,
and the arithmetic shortcuts the kernels rely on are exact."""
import ctypes as C
import re
from fractions import Fraction

import numpy as np
import pytest

import oracle_lib as ol
from sela_b200 import _lib


def test_library_exports_every_declared_symbol():
    header = _lib.HEADER_PATH.read_text()
    declared = set(re.findall(r"\b(selab200_[a-z0-9_]+)\s*\(", header))
    assert declared, "no entry points found in include/sela_b200.h"
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    L = _lib.lib()                      # dlopen + getattr of every symbol
    for name in declared:
        assert hasattr(L, name)
    assert L.selab200_abi_version() == 2


def test_descriptor_layout_matches_header_and_oracle():
    assert _lib.DESC_DTYPE.itemsize == 32 == ol.DESC_DTYPE.itemsize
    assert _lib.DESC_DTYPE == ol.DESC_DTYPE
    offs = {n: _lib.DESC_DTYPE.fields[n][1] for n in _lib.DESC_DTYPE.names}
    assert offs == {"channel": 0, "subframe_type": 1, "parent_channel": 2, "refl_rice_param": 3,
                    "refl_words": 4, "lpc_order": 6, "res_rice_param": 7, "res_words": 8, "samples": 10,
                    "reserved": 12, "refl_offset": 16, "res_offset": 24}


def test_no_cpu_fallback_without_device():
    """On a box without a GPU every compute entry point must fail loudly."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = _lib.lib()
    assert L.selab200_init(0) == -1
    assert b"no CPU path" in L.selab200_last_error()
    used = C.c_size_t(0)
    pcm = np.zeros(2048, np.int16)
    descs = np.zeros(1, _lib.DESC_DTYPE)
    words = np.zeros(4096, np.uint32)
    rc = L.selab200_encode_frames(pcm.ctypes.data, 1, 1, descs.ctypes.data, words.ctypes.data, 4096,
                                  C.addressof(used))
    assert rc == -7          # NOT_INIT: nothing silently computed on the CPU
    import sela_b200
    with pytest.raises(sela_b200.SelaB200Error):
        sela_b200.encode_frames(pcm, 1)


def test_workspace_and_bound_helpers():
    L = _lib.lib()
    assert L.selab200_encode_words_bound(10, 2) >= 10 * 2 * 1536
    assert L.selab200_encode_workspace_bytes(10, 2) >= 10 * 8
    assert L.selab200_decode_workspace_bytes(10, 2) >= 10 * 2 * (2048 + 128) * 4


def test_division_free_sample_scaling_is_exact():
    """sela_b200/csrc/lpc.cuh sample_to_x: q0 = s*rcp; r = fma(-q0, 32767, s); q = fma(r, rcp, q0)
    equals the correctly rounded s/32767 for EVERY s in the domain (emulated exactly)."""
    rcp = 1.0 / 32767.0

    def fma(a, b, c):
        return float(Fraction(a) * Fraction(b) + Fraction(c))

    for s in range(-65535, 65536):
        a = float(s)
        q0 = a * rcp
        r = fma(-q0, 32767.0, a)
        assert fma(r, rcp, q0) == a / 32767.0, s


def test_lpc_tables_identical_in_oracle_and_product():
    import pathlib
    root = pathlib.Path(__file__).resolve().parent.parent
    pat = re.compile(r"0x[0-9a-f]{16}ULL")
    a = pat.findall((root / "oracle" / "lpc_tables.inc").read_text())
    b = pat.findall((root / "sela_b200" / "csrc" / "lpc_tables.cuh").read_text())
    assert a == b and len(a) == 129
    # format constants match the reference header's firstOrderCoefficients[128], bit for bit
    bits = ol.golden("reference_stages")["lpc_first_order_bits"]
    assert ["0x%016xULL" % int(v) for v in bits] == a[:128]


def test_zero_history_bit_exactness_argument():
    """The autocorrelation kernel starts every lag's chain at j = 0 with d[negative] = +0.0
    instead of at j = i: acc + (+-0 * x) must leave acc = +0.0 unchanged, bitwise."""
    acc = np.float64(0.0)
    for x in (np.float64(3.5), np.float64(-2.25), np.float64(-0.0)):
        acc = acc + x * np.float64(0.0)
        assert acc.tobytes() == np.float64(0.0).tobytes()
