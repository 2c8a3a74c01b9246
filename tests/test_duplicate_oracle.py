"""Duplication bloom filter (SURVEY 8f rank 2, src/duplicate.cpp): the C port pinned against the reference's own Duplicate object.
Oracle first -- the device path is next round's work (DESIGN.md, "What comes next in 8f")."""
import ctypes as C

import numpy as np
import pytest

import fp_testlib as T
from fastp_b200 import capi

pytestmark = pytest.mark.reference


def planted(paired, n=4000, seed=9):
    """n units, then 40 % more drawn from them again (exact duplicates) plus a few one-base variants, shuffled."""
    rng = np.random.default_rng(seed)
    _, arrs = T.synth_host(n, 160, paired, 0, seed, 1, 150)
    pick = rng.integers(0, n, int(n * 0.4))
    out = {k: np.concatenate([v, v[pick]]) for k, v in arrs.items()}
    for i in rng.integers(n, len(out["len1"]), 60):              # near-duplicates: one substituted base
        if out["len1"][i] > 10:
            out["seq1"][i, 5] = ord("A") if out["seq1"][i, 5] != ord("A") else ord("C")
    perm = rng.permutation(len(out["len1"]))
    return {k: np.ascontiguousarray(v[perm]) for k, v in out.items()}


CUTS = lambda n: ((0, n // 3), (n // 3, n // 2), (n // 2, n))          # noqa: E731  (state carries over batches)


def _reference_duplicate(arrs, paired):
    """flags and (total, duplicated) of the reference's own Duplicate object over the batches of CUTS."""
    rlib = T.ref()
    rlib.fp_ref_dup_create.restype = C.c_void_p; rlib.fp_ref_dup_create.argtypes = [C.c_int]
    rlib.fp_ref_dup_check.argtypes = [C.c_void_p, C.POINTER(capi.Batch), C.c_int, C.c_void_p]
    rlib.fp_ref_dup_totals.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    rlib.fp_ref_dup_destroy.argtypes = [C.c_void_p]
    n = len(arrs["len1"])
    rd = rlib.fp_ref_dup_create(1)
    assert rd
    try:
        flags_r = np.zeros(n, np.uint8)
        for lo, hi in CUTS(n):
            b = capi.batch_from_arrays({k: np.ascontiguousarray(v[lo:hi]) for k, v in arrs.items()})
            fr = np.zeros(hi - lo, np.uint8)
            rlib.fp_ref_dup_check(rd, C.byref(b), paired, fr.ctypes.data)
            flags_r[lo:hi] = fr
        tr, dr, rate = C.c_int64(), C.c_int64(), C.c_double()
        rlib.fp_ref_dup_totals(rd, C.byref(tr), C.byref(dr), C.byref(rate))
        assert abs(rate.value - dr.value / n) < 1e-12
        return {"flags": flags_r, "totals": (tr.value, dr.value)}
    finally:
        rlib.fp_ref_dup_destroy(rd)


@pytest.mark.parametrize("paired", [1, 0])
def test_port_equals_reference_duplicate(paired):
    olib = T.oracle()
    olib.fp_oracle_dup_create.restype = C.c_void_p; olib.fp_oracle_dup_create.argtypes = [C.c_int]
    olib.fp_oracle_dup_check.argtypes = [C.c_void_p, C.POINTER(capi.Batch), C.c_int, C.c_void_p]
    olib.fp_oracle_dup_totals.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    olib.fp_oracle_dup_destroy.argtypes = [C.c_void_p]
    arrs = planted(paired)
    n = len(arrs["len1"])
    od = olib.fp_oracle_dup_create(1)
    assert od
    try:
        flags_o = np.zeros(n, np.uint8)
        for lo, hi in CUTS(n):
            b = capi.batch_from_arrays({k: np.ascontiguousarray(v[lo:hi]) for k, v in arrs.items()})
            fo = np.zeros(hi - lo, np.uint8)
            olib.fp_oracle_dup_check(od, C.byref(b), paired, fo.ctypes.data)
            flags_o[lo:hi] = fo
        to, do = C.c_int64(), C.c_int64()
        olib.fp_oracle_dup_totals(od, C.byref(to), C.byref(do))
        assert (to.value, do.value) == (n, int(flags_o.sum()))
        T.check_reference(f"duplicate/{paired}", {"flags": flags_o, "totals": (to.value, do.value)}, lambda: _reference_duplicate(arrs, paired))
        # every second copy of a planted exact duplicate is flagged (the filter has no false negatives)
        assert do.value >= int(n / 1.4 * 0.4) - 80
    finally:
        olib.fp_oracle_dup_destroy(od)


def _dup_positions(arrs, paired, buf_num=2, prime_len=512, buf_bits=(1 << 29) * 8):
    """Bit position of every unit in every array, vectorised restatement of seq2intvector (uint64 wrap-around arithmetic)."""
    primes = []
    number = 10000
    while len(primes) < buf_num * prime_len:
        number += 1
        if all(number % i for i in range(2, int(number ** 0.5) + 1)):
            primes.append(number); number += 10000
    primes = np.array(primes, np.uint64)
    lut = np.full(256, 13, np.uint64); lut[ord("A")] = 7; lut[ord("T")] = 222; lut[ord("C")] = 74; lut[ord("G")] = 31
    n = len(arrs["len1"])
    pos = np.zeros((n, buf_num), np.uint64)
    mask = buf_num * prime_len - 1
    with np.errstate(over="ignore"):
        for side, off in (("1", np.zeros(n, np.int64)), ("2", arrs["len1"].astype(np.int64)))[: 2 if paired else 1]:
            S = arrs["seq" + side].shape[1]
            p = np.arange(S)[None, :] + off[:, None]
            valid = np.arange(S)[None, :] < arrs["len" + side][:, None]
            base = lut[arrs["seq" + side]] + p.astype(np.uint64)
            for i in range(buf_num):
                w = primes[((p * buf_num + i) & mask)]
                pos[:, i] += np.where(valid, w * base, np.uint64(0)).sum(axis=1, dtype=np.uint64)
    return pos % np.uint64(buf_bits)


def test_first_toucher_formulation_equals_sequential_filter():
    """The device design (DESIGN.md): unit i is a duplicate iff, in every array, its bit is set from earlier batches or the smallest
    index touching that bit in this batch is < i.  Emulated with numpy and compared with the sequential C port, batch by batch."""
    olib = T.oracle()
    olib.fp_oracle_dup_create.restype = C.c_void_p; olib.fp_oracle_dup_create.argtypes = [C.c_int]
    olib.fp_oracle_dup_check.argtypes = [C.c_void_p, C.POINTER(capi.Batch), C.c_int, C.c_void_p]
    olib.fp_oracle_dup_destroy.argtypes = [C.c_void_p]
    for paired in (1, 0):
        arrs = planted(paired, n=3000, seed=21 + paired)
        n = len(arrs["len1"])
        od = olib.fp_oracle_dup_create(1)
        try:
            persistent = [set(), set()]
            for lo, hi in ((0, n // 2), (n // 2, n)):
                sub = {k: np.ascontiguousarray(v[lo:hi]) for k, v in arrs.items()}
                b = capi.batch_from_arrays(sub)
                want = np.zeros(hi - lo, np.uint8)
                olib.fp_oracle_dup_check(od, C.byref(b), paired, want.ctypes.data)
                pos = _dup_positions(sub, paired)
                m = hi - lo
                got = np.ones(m, bool)
                for a in range(2):
                    first = {}
                    for i in range(m):                                   # pass 1: first toucher of every bit (atomicMin on the device)
                        first.setdefault(int(pos[i, a]), i)
                    for i in range(m):                                   # pass 2
                        k = int(pos[i, a])
                        got[i] &= (k in persistent[a]) or first[k] < i
                    persistent[a].update(first)                           # pass 3
                assert np.array_equal(got.astype(np.uint8), want), (paired, lo)
        finally:
            olib.fp_oracle_dup_destroy(od)


def test_device_bodies_emulated_on_host_equal_the_oracle(tmp_path):
    """fastp_b200/csrc/fp_dup.h holds the per-thread bodies of the device passes as host+device functions; here they run on the host,
    one thread at a time in shuffled order, over three batches -- same flags as the sequential C port, whatever the order."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "dup_emulation"
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(root, "fastp_b200", "csrc"), os.path.join(root, "tests", "host", "dup_emulation.cpp"),
                    "-o", str(exe)], check=True)
    olib = T.oracle()
    olib.fp_oracle_dup_create.restype = C.c_void_p; olib.fp_oracle_dup_create.argtypes = [C.c_int]
    olib.fp_oracle_dup_check.argtypes = [C.c_void_p, C.POINTER(capi.Batch), C.c_int, C.c_void_p]
    olib.fp_oracle_dup_destroy.argtypes = [C.c_void_p]
    for paired in (1, 0):
        arrs = planted(paired, n=3000, seed=33 + paired)
        n = len(arrs["len1"])
        cuts = [(0, n // 3), (n // 3, n // 2), (n // 2, n)]
        path = tmp_path / f"b{paired}.bin"
        od = olib.fp_oracle_dup_create(1)
        want = []
        try:
            with open(path, "wb") as f:
                f.write(np.int64(len(cuts)).tobytes())
                for lo, hi in cuts:
                    sub = {k: np.ascontiguousarray(v[lo:hi]) for k, v in arrs.items()}
                    f.write(np.int64(hi - lo).tobytes()); f.write(np.int32(160).tobytes()); f.write(np.int32(paired).tobytes())
                    f.write(sub["seq1"].tobytes()); f.write(sub["len1"].tobytes())
                    if paired:
                        f.write(sub["seq2"].tobytes()); f.write(sub["len2"].tobytes())
                    b = capi.batch_from_arrays(sub)
                    w = np.zeros(hi - lo, np.uint8)
                    olib.fp_oracle_dup_check(od, C.byref(b), paired, w.ctypes.data)
                    want.append("".join(map(str, w)))
        finally:
            olib.fp_oracle_dup_destroy(od)
        for seed in (1, 2):
            got = subprocess.run([str(exe), str(path), "1", str(seed)], check=True, capture_output=True, text=True).stdout.strip().split("\n")
            assert got == want, (paired, seed)
        assert sum(x.count("1") for x in want) > 500
