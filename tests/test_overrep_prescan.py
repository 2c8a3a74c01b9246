"""Host pre-scan of the over-representation candidates (fp_host_overrep_candidates, control plane of BASELINE configs[4]) against
the reference's own Evaluator::computeOverRepSeq (src/evaluator.cpp:78-169), compiled from its sources into oracle/_ref."""
import ctypes as C
import os

import numpy as np
import pytest

import fp_testlib as T
from fastp_b200 import capi


def host_candidates(seq, lens, stride, seqlen):
    lib = capi.load()
    out = C.create_string_buffer(1 << 22); n = C.c_int32(); used = C.c_int64()
    rc = lib.fp_host_overrep_candidates(np.ascontiguousarray(seq).ctypes.data, np.ascontiguousarray(lens).ctypes.data, seq.shape[0], stride, seqlen,
                                        out, len(out), C.byref(n), C.byref(used))
    assert rc == 0
    c = out.raw[:used.value].split(b"\0")[:-1]
    assert len(c) == n.value
    return c


def reference_candidates(tmp_path, arrs, side, L):
    """Evaluator::computeOverRepSeq of the reference over the same reads written as FASTQ."""
    ref = T.ref()
    ref.fp_ref_compute_overrep.restype = C.c_int
    ref.fp_ref_compute_overrep.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    fn = os.path.join(tmp_path, f"r{side}.fq")
    open(fn, "wb").write(T.fastq_text(arrs["seq" + side], arrs["qual" + side], arrs["len" + side], side))
    out = C.create_string_buffer(1 << 22); used = C.c_int64()
    k = ref.fp_ref_compute_overrep(fn.encode(), L, out, len(out), C.byref(used))
    want = out.raw[:used.value].split(b"\0")[:-1]
    assert k == len(want)
    return want


@pytest.mark.parametrize("L,S,profile,n", [(250, 256, 3, 7000), (150, 160, 1, 4000), (100, 112, 3, 3000)])
def test_candidates_equal_reference_evaluator(tmp_path, L, S, profile, n):
    _, arrs = T.synth_host(n, S, 1, 0, 42, profile, L)
    for side in "12":
        got = host_candidates(arrs["seq" + side], arrs["len" + side], S, L)
        T.check_reference(f"overrep_prescan/{L}/{side}", got, lambda: reference_candidates(tmp_path, arrs, side, L))
    if profile == 3:
        assert len(got) > 0          # the planted sequences are found


def test_small_buffer_reports_size():
    _, arrs = T.synth_host(3000, 256, 1, 0, 42, 3, 250)
    lib = capi.load()
    n = C.c_int32(); used = C.c_int64()
    rc = lib.fp_host_overrep_candidates(arrs["seq1"].ctypes.data, arrs["len1"].ctypes.data, 3000, 256, 250, None, 0, C.byref(n), C.byref(used))
    assert (rc == 0 and used.value == 0) or rc == -4     # FP_E_TOOLARGE with the size needed
    if rc != 0:
        assert used.value > 0 and n.value > 0
