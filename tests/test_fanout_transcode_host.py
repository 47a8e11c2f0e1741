"""The G.711 code table of igd_gateway_fanout_packets (igd_g711_transcode1 in csrc/igd_math.cuh, built for the host
with -DIGD_HOST_EMUL), checked entry by entry against the oracle's decode then encode."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_py as O

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostbuild", "transcode_emul.cpp")
CODES = np.arange(256, dtype=np.uint8)


@pytest.fixture(scope="module")
def table(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("transcode") / "libtranscode.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", so, SRC])
    out = np.zeros((2, 2, 256), np.uint8)           # [in law][out law][code], 0 = A-law, 1 = u-law
    C.CDLL(so).emul_transcode_table(C.c_void_p(out.ctypes.data))
    return out


@pytest.mark.parametrize("in_law", [0, 1])
@pytest.mark.parametrize("out_law", [0, 1])
def test_every_entry_is_decode_then_encode(table, in_law, out_law):
    want = O.g711_encode(O.g711_decode(CODES, in_law), out_law)
    assert np.array_equal(table[in_law, out_law], want)


def test_same_law_identities(table):
    assert np.array_equal(table[0, 0], CODES)                  # A-law -> A-law
    want = CODES.copy()
    want[0x7F] = 0xFF                                          # u-law -0 -> +0
    assert np.array_equal(table[1, 1], want)
    # u-law 0xFF decodes to PCM 0: its row entries are the silence codes the kernel sends for a tick without audio
    assert O.g711_decode(np.array([0xFF], np.uint8), 1)[0] == 0
    assert (table[1, 0, 0xFF], table[1, 1, 0xFF]) == (0xD5, 0xFF)
