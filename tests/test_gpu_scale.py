"""-m gpu parity at the survey's scale (SURVEY.md 8d: per-read records + all counters bit-exact on the first >= 10 M units of each
config): the CUDA path against the REFERENCE's own worker body (oracle/_ref: the reference's objects compiled from its sources),
run on all host threads.  The reference's counter block is thread-count invariant for these option sets (SURVEY App. C: the harness
gives every worker thread-0 semantics), the per-read records are per unit anyway."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

import fp_testlib as T
from fastp_b200 import capi

pytestmark = pytest.mark.gpu
UNITS = int(os.environ.get("FP_SCALE_UNITS", 10_000_000))


def synth_parallel(n, S, paired, profile, L, threads):
    b, arrs = capi.host_batch(n, S, paired)
    lib = T.oracle()
    bounds = [n * i // threads for i in range(threads + 1)]

    def work(i):
        lo, hi = bounds[i], bounds[i + 1]
        if hi > lo:
            sb = capi.batch_from_arrays({k: v[lo:hi] for k, v in arrs.items()})
            lib.fp_synth_fill_host(C.byref(sb), lo, 42, profile, L)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    [t.start() for t in ts]; [t.join() for t in ts]
    return arrs


def reference_fields(p, arrs, paired, threads):
    """records + counters + corrected rows of the reference's worker body over a copy of the rows, on `threads` host threads."""
    n, S = arrs["seq1"].shape
    a = {k: v.copy() for k, v in arrs.items()}
    rb = capi.batch_from_arrays(a)
    Lr = capi.make_layout(T.oracle(), paired, S, p.insert_size_max)
    want_cnt = np.zeros(Lr.total, np.int64)
    w1 = np.zeros(n, capi.READ_RESULT_DTYPE); w2 = np.zeros(n, capi.READ_RESULT_DTYPE); wov = np.zeros(n, capi.OV_RESULT_DTYPE)
    rc = T.ref().fp_ref_process_mt(C.byref(p), C.byref(Lr), C.byref(rb), w1.ctypes.data, w2.ctypes.data if paired else None,
                                   wov.ctypes.data if paired else None, want_cnt.ctypes.data, threads)
    assert rc == 0
    want = {"out1": w1, "out2": w2, "ov": wov, "counters": capi.CounterView(Lr, want_cnt), "arrs": a}
    # adapter_pos is a device-side extra (where trimBySequence hit); the reference harness has no such field
    return T.result_fields(want, paired, skip=("adapter_pos",))


CASES = [("cfg2_cut_right_polyg", 0), ("cfg3_overlap_correction", 1), ("cfg4_full", 1)]


@pytest.mark.parametrize("name,paired", CASES)
def test_ten_million_units_equal_reference(name, paired):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("CUDA device required for -m gpu tests (no CPU fallback exists)")
    import fp_gpu
    n, S, L = UNITS, 160, 150
    threads = len(os.sched_getaffinity(0))
    arrs = synth_parallel(n, S, paired, 1, L, min(threads, 32))
    p = T.config_params(name, paired, lib=T.oracle())
    # CUDA: HBM-resident, one launch
    ctx = fp_gpu.GpuCtx(p, 1 << 18, S, S)
    t = {k: torch.from_numpy(v).cuda() for k, v in arrs.items()}
    b = capi.Batch(); b.n, b.stride = n, S
    for k, v in t.items():
        setattr(b, k, v.data_ptr())
    o1 = torch.zeros(n * 16, dtype=torch.uint8, device="cuda:0"); o2 = torch.zeros(n * 16 if paired else 16, dtype=torch.uint8, device="cuda:0")
    ov = torch.zeros(n * 8 if paired else 8, dtype=torch.uint8, device="cuda:0")
    if paired:
        capi.check(ctx.lib.fp_process_pe(ctx.h, C.byref(b), o1.data_ptr(), o2.data_ptr(), ov.data_ptr(), None, 0, None, None), ctx.lib)
    else:
        capi.check(ctx.lib.fp_process_se(ctx.h, C.byref(b), o1.data_ptr(), None), ctx.lib)
    torch.cuda.synchronize()
    got = {"out1": o1.cpu().numpy().view(capi.READ_RESULT_DTYPE), "out2": o2.cpu().numpy().view(capi.READ_RESULT_DTYPE)[:n if paired else 0],
           "ov": ov.cpu().numpy().view(capi.OV_RESULT_DTYPE)[:n if paired else 0], "counters": ctx.counters(),
           "arrs": {k: v.cpu().numpy().reshape(arrs[k].shape) for k, v in t.items()}}
    ctx.close()
    del t
    T.check_reference(f"scale/{name}/{n}", T.result_fields(got, paired, skip=("adapter_pos",)), lambda: reference_fields(p, arrs, paired, threads))
