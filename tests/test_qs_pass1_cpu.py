"""The fused qshmm pass 1 of the kernels (qshmm_chunk_pass1, run by k_qs_pass1) against the split statement the CPU
harness runs (qshmm_quality_range + qshmm_error_segment), which the other CPU tests compare with the oracle: event
slots and segment results must be equal, byte for byte, compiled as plain C++ (no GPU)."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest

from pbsim_b200 import capi
from tests.golden_util import model_path

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def lib():
    out = tempfile.mkdtemp(prefix="qs_pass1_check_")
    so = os.path.join(out, "libqs_pass1_check.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", so,
                           os.path.join(HERE, "hostsim", "qs_pass1_check.cpp"),
                           os.path.join(ROOT, "pbsim_b200", "csrc", "host_model.cpp")])
    L = C.CDLL(so)
    capi.declare_host(L)
    L.qs_pass1_compare.restype = C.c_long
    L.qs_pass1_compare.argtypes = [C.POINTER(capi.Model), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                   C.POINTER(C.c_long)]
    return L


@pytest.mark.parametrize("model", ["QSHMM-ONT.model", "QSHMM-RSII.model"])
@pytest.mark.parametrize("chunk", [0, 1, 3])
@pytest.mark.parametrize("del_floor", [0, 0x99999999])
def test_fused_pass1_equals_split_passes(lib, model, chunk, del_floor):
    """every accuracy with a chain, chunks of 1 and 3 segments and whole reads; with del_floor the deletion
    thresholds are raised to 0.6 so that the >= 15-deletion redo and leading insertions are common"""
    hm = capi.HostModel(lib, capi.host_params("qshmm"), model_path(model))
    try:
        stats = (C.c_long * 4)()
        bad = lib.qs_pass1_compare(hm.ptr, 7, 3, 5, chunk, del_floor, stats)
    finally:
        hm.close()
    assert bad == 0 and stats[3] == 0
    assert stats[0] > 100
    if del_floor:
        assert stats[1] > 0, "no segment was redone generically"
        assert stats[2] > 0, "no read started with an insertion"
