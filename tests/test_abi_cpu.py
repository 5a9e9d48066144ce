"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, exports every
symbol include/*.h declares, refuses to run without a GPU (no CPU fallback), and its constant tables
equal the oracle's (which are pinned to the reference's literal arrays)."""
import ctypes as C
import glob
import os
import re

import numpy as np
import pytest

import h264lib

ROOT = h264lib.ROOT


@pytest.fixture(scope="module")
def L():
    import openh264_b200 as m
    m.build()
    return m.load()


def declared_symbols():
    names = set()
    for hdr in glob.glob(os.path.join(ROOT, "include", "*.h")):
        txt = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)
        names |= set(re.findall(r"\b((?:b2h264_|Wels)\w+)\s*\(", txt))
    return sorted(names)


def test_every_declared_symbol_is_exported(L):
    # layers 1-2 (b2h264_*) live in libopenh264_b200.so; layer 3 (the reference's own Wels* entry points,
    # include/b2h264_wels_api.h) in libopenh264_b200_wels.so, which links against the former
    import ctypes
    wels_so = os.path.join(ROOT, "openh264_b200", "libopenh264_b200_wels.so")
    assert os.path.exists(wels_so), "build() makes it"
    Wl = ctypes.CDLL(wels_so)
    missing = [n for n in declared_symbols() if not hasattr(Wl if n.startswith("Wels") else L, n)]
    assert not missing, missing
    assert len(declared_symbols()) > 30


def test_python_binding_covers_header():
    from openh264_b200.binding import API
    assert set(n for n in declared_symbols() if n.startswith("b2h264_")) <= set(API)


def test_abi_version(L):
    assert L.b2h264_abi_version() == 1


def test_no_cpu_fallback(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert L.b2h264_init(0) != 0          # fails loudly: no device, no fallback
    import openh264_b200 as m
    with pytest.raises(m.B2H264Error):
        m.lib.__globals__["_inited"] = False
        m.lib(0)


def test_tables_match_oracle(L):
    orc = h264lib.oracle()
    for q in range(58):
        assert np.array_equal(np.ctypeslib.as_array(L.b2h264_table_quant_ff(q), shape=(8,)),
                              np.ctypeslib.as_array(orc.quant_ff(q), shape=(8,)))
    for q in range(52):
        assert np.array_equal(np.ctypeslib.as_array(L.b2h264_table_quant_mf(q), shape=(8,)),
                              np.ctypeslib.as_array(orc.quant_mf(q), shape=(8,)))
        assert np.array_equal(np.ctypeslib.as_array(L.b2h264_table_dequant(q), shape=(8,)),
                              np.ctypeslib.as_array(orc.dequant_coeff(q), shape=(8,)))
        assert L.b2h264_table_lambda(q) == orc.qp_lambda(q)
        assert L.b2h264_table_chroma_qp(q) == orc.chroma_qp(q)
