"""Test infrastructure: loaders for the CPU checkers under oracle/ and comparison helpers.
Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may use oracle/."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

from fastp_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "libfastp_oracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libfastp_ref.so")
REF_CLI = os.path.join(ORACLE_DIR, "_ref", "fastp_ref")

TRUSEQ_R1 = "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA"
TRUSEQ_R2 = "AGATCGGAAGAGCGTCGTGTAGGGAAAGAGTGT"

_PROC_ARGS = [C.POINTER(capi.Params), C.POINTER(capi.CounterLayout), C.POINTER(capi.Batch),
              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]

_oracle = None
_ref = None


def build_oracle():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "libfastp_oracle.so"], check=True)


def oracle():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        lib = C.CDLL(ORACLE_SO)
        capi.bind(lib, ["fp_params_default", "fp_counter_layout_make", "fp_counter_layout_make_overrep", "fp_abi_sizeof"])
        lib.fp_oracle_process.restype = C.c_int
        lib.fp_oracle_process.argtypes = _PROC_ARGS
        lib.fp_synth_fill_host.restype = C.c_int
        lib.fp_synth_fill_host.argtypes = [C.POINTER(capi.Batch), C.c_int64, C.c_uint64, C.c_int32, C.c_int32]
        lib.fp_oracle_trim_and_cut.restype = C.c_int
        lib.fp_oracle_trim_and_cut.argtypes = [C.POINTER(capi.Params), C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int,
                                               C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.fp_oracle_trim_polyg.restype = C.c_int
        lib.fp_oracle_trim_polyg.argtypes = [C.c_char_p, C.c_int, C.c_int]
        lib.fp_oracle_trim_polyx.restype = C.c_int
        lib.fp_oracle_trim_polyx.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.fp_oracle_trim_by_sequence.restype = C.c_int
        lib.fp_oracle_trim_by_sequence.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.POINTER(C.c_int)]

        class OV(C.Structure):
            _fields_ = [("overlapped", C.c_uint8), ("has_gap", C.c_uint8), ("offset", C.c_int16),
                        ("overlap_len", C.c_int16), ("diff", C.c_int16)]
        lib.fp_oracle_analyze.restype = OV
        lib.fp_oracle_analyze.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_double]
        lib.fp_oracle_pass_filter.restype = C.c_int
        lib.fp_oracle_pass_filter.argtypes = [C.POINTER(capi.Params), C.c_char_p, C.c_char_p, C.c_int]
        lib.fp_oracle_match_with_one_insertion.restype = C.c_int
        lib.fp_oracle_match_with_one_insertion.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        _oracle = lib
    return _oracle


def have_ref():
    return os.path.exists(REF_SO)


def ref():
    global _ref
    if _ref is None:
        lib = C.CDLL(REF_SO)
        lib.fp_ref_process.restype = C.c_int
        lib.fp_ref_process.argtypes = _PROC_ARGS
        lib.fp_ref_process_mt.restype = C.c_int
        lib.fp_ref_process_mt.argtypes = _PROC_ARGS + [C.c_int]
        _ref = lib
    return _ref


# ---------------- the reference's answers, stored as digests ----------------
# oracle/_ref is built only where the reference sources are.  Every comparison with it is therefore pinned by the digests of the
# reference's answers in REF_DIGESTS: without the build the tested value must hash to them; with it the reference runs as well,
# its answer must still hash to them (FP_UPDATE_GOLDEN=1 rewrites them instead) and the tested value must equal it.
REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")
_digests = None


def _feed(h, o):
    if isinstance(o, np.ndarray):
        h.update(repr((o.dtype.str, o.shape)).encode())
        h.update(np.ascontiguousarray(o).tobytes())
    elif isinstance(o, dict):
        h.update(b"{%d" % len(o))
        for k in sorted(o):
            _feed(h, k); _feed(h, o[k])
    elif isinstance(o, (list, tuple)):
        h.update(b"[%d" % len(o))
        for x in o:
            _feed(h, x)
    elif isinstance(o, bytes):
        h.update(b"b%d:" % len(o)); h.update(o)
    else:
        h.update(repr(o.item() if isinstance(o, np.generic) else o).encode())


def digest(obj):
    h = hashlib.sha256()
    _feed(h, obj)
    return h.hexdigest()[:12]


def _digest_of(obj):
    return {k: digest(v) for k, v in obj.items()} if isinstance(obj, dict) else digest(obj)


def _assert_same(got, want, what):
    if isinstance(want, dict):
        assert sorted(got) == sorted(want), f"{what}: keys {sorted(got)} vs {sorted(want)}"
        for k in want:
            _assert_same(got[k], want[k], f"{what}.{k}")
    elif isinstance(want, np.ndarray):
        assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
        i = np.argwhere(got != want)
        assert i.size == 0, f"{what} differs at {tuple(i[0])}: {got[tuple(i[0])]} vs {want[tuple(i[0])]}"
    else:
        assert got == want, f"{what}: {got!r} vs {want!r}"


def check_reference(key, got, reference):
    """Assert that `got` equals the reference's answer for case `key`; reference() computes that answer with oracle/_ref.
    A dict is pinned key by key, so a failure names the field."""
    global _digests
    if _digests is None:
        _digests = json.load(open(REF_DIGESTS)) if os.path.exists(REF_DIGESTS) else {}
    if have_ref():
        want = reference()
        if os.environ.get("FP_UPDATE_GOLDEN") == "1":
            _digests[key] = _digest_of(want)
            with open(REF_DIGESTS, "w") as f:
                json.dump(_digests, f, indent=0, sort_keys=True)
                f.write("\n")
        else:
            assert _digest_of(want) == _digests.get(key), f"{key}: the reference's answer no longer matches {REF_DIGESTS} (FP_UPDATE_GOLDEN=1 rewrites it)"
        _assert_same(got, want, key)
        return
    assert key in _digests, f"{key}: no stored reference answer in {REF_DIGESTS}"
    stored, mine = _digests[key], _digest_of(got)
    if isinstance(stored, dict):
        assert sorted(mine) == sorted(stored), f"{key}: fields {sorted(mine)} vs {sorted(stored)}"
        bad = [k for k in stored if mine[k] != stored[k]]
        assert not bad, f"{key}: {', '.join(bad)} differ from the reference's"
    else:
        assert mine == stored, f"{key}: differs from the reference's answer"


def result_fields(res, paired, skip=()):
    """The fields assert_results_equal compares, as one dict of arrays: records, overlap records, corrected rows (bytes past a
    read's length zeroed) and the counter block."""
    out = {}
    for o in ("out1", "out2") if paired else ("out1",):
        for f in RESULT_FIELDS:
            if f not in skip:
                out[f"{o}.{f}"] = np.ascontiguousarray(res[o][f])
    if paired and "ov" not in skip:
        for f in ("overlapped", "has_gap", "offset", "overlap_len", "diff"):
            out[f"ov.{f}"] = np.ascontiguousarray(res["ov"][f])
    for k, a in res["arrs"].items():
        if not k.startswith("len"):
            ln = res["arrs"]["len" + k[-1]].astype(np.int64)
            out[k] = np.where(np.arange(a.shape[1])[None, :] < ln[:, None], a, 0).astype(a.dtype)
    out["counters"] = res["counters"].data
    return out


def check_result_reference(key, got, params, arrs, cycles, skip=(), nthreads=0):
    """check_reference for a run_cpu / run_gpu result: the reference harness over the same batch is the answer."""
    paired = bool(params.paired)
    check_reference(key, result_fields(got, paired, skip),
                    lambda: result_fields(run_cpu("ref", params, arrs, cycles, nthreads), paired, skip))


def copy_arrays(arrs):
    return {k: v.copy() for k, v in arrs.items()}


def synth_host(n, stride, paired, first_index, seed, profile, read_len):
    b, arrs = capi.host_batch(n, stride, paired)
    rc = oracle().fp_synth_fill_host(C.byref(b), first_index, seed, profile, read_len)
    assert rc == 0
    return b, arrs


def run_cpu(which, params, arrs, cycles, nthreads=0):
    """Run the C port ('oracle') or the reference harness ('ref') over a COPY of arrs.
    Returns dict(out1, out2, ov, counters(CounterView), arrs(after correction))."""
    a = copy_arrays(arrs)
    b = capi.batch_from_arrays(a)
    paired = bool(params.paired)
    L = capi.make_layout(oracle(), paired, cycles, params.insert_size_max, params)
    n = b.n
    out1 = np.zeros(n, capi.READ_RESULT_DTYPE)
    out2 = np.zeros(n, capi.READ_RESULT_DTYPE)
    ov = np.zeros(n, capi.OV_RESULT_DTYPE)
    cnt = np.zeros(L.total, np.int64)
    args = (C.byref(params), C.byref(L), C.byref(b), out1.ctypes.data, out2.ctypes.data if paired else None,
            ov.ctypes.data if paired else None, cnt.ctypes.data)
    if which == "oracle":
        rc = oracle().fp_oracle_process(*args)
    elif nthreads:
        rc = ref().fp_ref_process_mt(*args, nthreads)
    else:
        rc = ref().fp_ref_process(*args)
    assert rc == 0, rc
    return {"out1": out1, "out2": out2, "ov": ov, "counters": capi.CounterView(L, cnt), "arrs": a, "layout": L}


RESULT_FIELDS = ("front", "len", "verdict", "flags", "adapter_pos", "adapter_len", "polyx_base", "pair_verdict", "polyx_len")


def first_diff(a, b):
    idx = np.nonzero(a != b)[0]
    return int(idx[0]) if idx.size else -1


def assert_results_equal(x, y, paired, skip=(), what=""):
    """Bit-exact comparison of per-read records, overlap records, corrected bases and all counters."""
    outs = ("out1", "out2") if paired else ("out1",)
    for o in outs:
        for f in RESULT_FIELDS:
            if f in skip:
                continue
            xa, ya = x[o][f], y[o][f]
            if f in ("front", "len") :
                # a dropped read (trimAndCut -> NULL) has no window
                pass
            i = first_diff(xa, ya)
            assert i < 0, f"{what} {o}.{f} differs at read {i}: {xa[i]} vs {ya[i]} (rec {x[o][i]} vs {y[o][i]})"
    if paired and "ov" not in skip:
        for f in ("overlapped", "has_gap", "offset", "overlap_len", "diff"):
            i = first_diff(x["ov"][f], y["ov"][f])
            assert i < 0, f"{what} ov.{f} differs at pair {i}: {x['ov'][i]} vs {y['ov'][i]}"
    for k in x["arrs"]:
        if k.startswith("len"):
            continue
        i = first_diff((x["arrs"][k] != y["arrs"][k]).any(axis=1), np.zeros(x["arrs"][k].shape[0], bool))
        if i >= 0:
            # only the valid part of the row matters
            ln = x["arrs"]["len" + k[-1]][i]
            assert (x["arrs"][k][i, :ln] == y["arrs"][k][i, :ln]).all(), f"{what} {k} row {i} differs after correction"
    assert_counters_equal(x["counters"], y["counters"], what)


def assert_counters_equal(cx, cy, what=""):
    L = cx.L
    assert cx.data.size == cy.data.size
    if (cx.data == cy.data).all():
        return
    names = {0: "pre1", 1: "post1", 2: "pre2", 3: "post2"}
    for s in range(L.n_stats):
        sx, sy = cx.stats(s), cy.stats(s)
        for key in ("cycle", "kmer", "qualhist"):
            if not (sx[key] == sy[key]).all():
                idx = np.argwhere(sx[key] != sy[key])[0]
                raise AssertionError(f"{what} stats[{names[s]}].{key}{tuple(idx)}: {sx[key][tuple(idx)]} vs {sy[key][tuple(idx)]}")
        for key in ("reads", "length_sum"):
            assert sx[key] == sy[key], f"{what} stats[{names[s]}].{key}: {sx[key]} vs {sy[key]}"
    for s in range(L.n_stats):
        (xc, xd), (yc, yd) = cx.overrep(s), cy.overrep(s)
        if not (xc == yc).all():
            i = int(np.nonzero(xc != yc)[0][0])
            raise AssertionError(f"{what} stats[{names[s]}].overrep_count[{i}]: {xc[i]} vs {yc[i]}")
        if not (xd == yd).all():
            idx = np.argwhere(xd != yd)[0]
            raise AssertionError(f"{what} stats[{names[s]}].overrep_dist{tuple(idx)}: {xd[tuple(idx)]} vs {yd[tuple(idx)]}")
    if not (cx.filter == cy.filter).all():
        i = int(np.nonzero(cx.filter != cy.filter)[0][0])
        raise AssertionError(f"{what} filter[{i}]: {cx.filter[i]} vs {cy.filter[i]}")
    if not (cx.isize == cy.isize).all():
        i = int(np.nonzero(cx.isize != cy.isize)[0][0])
        raise AssertionError(f"{what} isize[{i}]: {cx.isize[i]} vs {cy.isize[i]}")
    raise AssertionError(f"{what} counter blocks differ")


# Parameter sets exercised by the parity tests (names follow the fastp CLI flags they model).
def config_params(name, paired, lib=None):
    lib = lib or oracle()
    P = lambda **kw: capi.default_params(paired, lib=lib, **kw)  # noqa: E731
    if name.startswith("gap_"):               # --allow_gap_overlap_trimming on top of a base option set
        p = config_params(name[4:], paired, lib)
        capi.set_params(p, allow_gap_overlap_trimming=1)
        return p
    if name.startswith("merge_") or name.startswith("mergeu_"):   # --merge (forces --correction, options.cpp:120-121) [+ --include_unmerged]
        p = config_params(name.split("_", 1)[1], paired, lib)
        capi.set_params(p, merge_enabled=1, correction_enabled=1, merge_include_unmerged=1 if name.startswith("mergeu_") else 0)
        return p
    if name == "tight_overlap":               # stricter overlap thresholds + correction + gap passes
        return P(correction_enabled=1, allow_gap_overlap_trimming=1, overlap_require=20, overlap_diff_limit=3,
                 overlap_diff_percent_limit=10, adapter_seq_r1=TRUSEQ_R1, adapter_seq_r2=TRUSEQ_R2)
    if name == "default":
        return P()
    if name == "cfg2_cut_right_polyg":        # BASELINE config 2: --cut_right --trim_poly_g -A
        return P(cut_right=1, polyg_enabled=1, adapter_enabled=0)
    if name == "cfg3_overlap_correction":     # BASELINE config 3: overlap adapter trimming + --correction
        return P(correction_enabled=1)
    if name == "cfg4_full":                   # BASELINE config 4: --cut_right -g -x -c + adapter seqs
        return P(cut_right=1, polyg_enabled=1, polyx_enabled=1, correction_enabled=1,
                 adapter_seq_r1=TRUSEQ_R1, adapter_seq_r2=TRUSEQ_R2)
    if name == "cut_front_tail":
        return P(cut_front=1, cut_tail=1, cut_front_window=4, cut_front_quality=20, cut_tail_window=5, cut_tail_quality=18)
    if name == "trim_fixed":
        return P(trim_front1=3, trim_tail1=2, trim_front2=5, trim_tail2=1, max_len1=100, max_len2=90)
    if name == "all_cuts":
        return P(cut_front=1, cut_right=1, cut_tail=1, trim_front1=2, trim_tail2=3, cut_right_window=6, cut_right_quality=25,
                 polyx_enabled=1, polyg_enabled=1, polyx_min_len=8, polyg_min_len=12,
                 adapter_seq_r1=TRUSEQ_R1, adapter_seq_r2=TRUSEQ_R2)
    if name == "filters":
        return P(complexity_filter_enabled=1, complexity_threshold=30 / 100.0, avg_qual_req=25, length_required=40,
                 length_limit=148, n_base_limit=2, unqualified_percent_limit=20, qualified_qual=ord('5'))
    if name == "no_filters":
        return P(qual_filter_enabled=0, length_filter_enabled=0, adapter_enabled=0)
    if name == "fasta_adapters":
        return P(fasta_adapters=[TRUSEQ_R1, "CTGTCTCTTATACACATCT", TRUSEQ_R2[:20], "AAAAAAAAAAAA", "GGGGGGGGGG"],
                 adapter_seq_r1=TRUSEQ_R1[:12])
    if name == "tid_nonzero":
        return P(thread0_semantics=0, adapter_enabled=0)
    if name == "short_adapter":
        return P(adapter_seq_r1="AGATCGGAAG", adapter_seq_r2="AGATCGG", polyx_enabled=1)
    raise KeyError(name)


def overrep_candidates(arrs, side, L, seed=1, per_step=6):
    """Candidate list for over-representation tests: substrings of the batch itself at the five step lengths the
    reference scans (stats.cpp:274), plus candidates that can never match (wrong length) or match by chance."""
    rng = np.random.default_rng(seed)
    out = set()
    n = arrs["seq" + side].shape[0]
    for step in (10, 20, 40, 100, min(150, L - 2)):
        for _ in range(per_step):
            r = int(rng.integers(0, n)); ln = int(arrs["len" + side][r])
            if ln > step + 1:
                i = int(rng.integers(0, ln - step))
                out.add(bytes(arrs["seq" + side][r, i:i + step]).decode())
    out.update(["ACGTACGTAC", "G" * 20, "A" * 15, "G" * 10, "A" * 10])
    return sorted(out)


def overrep_params(name, paired, arrs, L, sampling=20, lib=None):
    p = config_params(name, paired, lib)
    kw = dict(overrep_enabled=1, overrep_sampling=sampling, seq_len1=L, seq_len2=L, overrep_seqs1=overrep_candidates(arrs, "1", L))
    if paired:
        kw["overrep_seqs2"] = overrep_candidates(arrs, "2", L, seed=2)
    capi.set_params(p, **kw)
    return p


CONFIG_NAMES = ["default", "cfg2_cut_right_polyg", "cfg3_overlap_correction", "cfg4_full", "cut_front_tail", "trim_fixed",
                "all_cuts", "filters", "no_filters", "fasta_adapters", "tid_nonzero", "short_adapter"]
# option sets for the one-gap overlap passes; run on synthetic profile 2 (reads with single-base indels)
MERGE_CONFIG_NAMES = ["merge_default", "merge_cfg4_full", "mergeu_cfg3_overlap_correction", "merge_filters", "mergeu_all_cuts", "merge_trim_fixed",
                      "mergeu_gap_cfg4_full"]
GAP_CONFIG_NAMES = ["gap_default", "gap_cfg3_overlap_correction", "gap_cfg4_full", "gap_all_cuts", "tight_overlap"]


# ---------------- FASTQ text <-> rows (SURVEY 8f rank 1) ----------------
def fastq_text(seq, qual, lens, tag, eol="\n", strand="+"):
    """FASTQ text of one side of a batch (names as the reference's benchmark generator writes them)."""
    out = []
    for i in range(seq.shape[0]):
        n = int(lens[i])
        out.append(f"@SIM:1:{i} {tag}{eol}{bytes(seq[i, :n]).decode()}{eol}{strand}{eol}{bytes(qual[i, :n]).decode()}{eol}")
    return "".join(out).encode()


def _bind_fastq(lib):
    if getattr(lib, "_fq_bound", False):
        return
    lib.fp_oracle_fastq_decode.restype = C.c_int
    lib.fp_oracle_fastq_decode.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_void_p, C.POINTER(capi.FastqInfo)]
    lib.fp_oracle_fastq_encode.restype = C.c_int64
    lib.fp_oracle_fastq_encode.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int64]
    lib._fq_bound = True


def info_dict(info):
    return {k: int(getattr(info, k)) for k, _ in capi.FastqInfo._fields_}


def oracle_fastq_decode(text, final=1, phred64=0, stride=160, capacity=None):
    """CPU oracle (FastqReader::read restated): rows, lens, records, info of one chunk."""
    lib = oracle(); _bind_fastq(lib)
    cap = capacity if capacity is not None else text.count(b"@") + 2
    buf = np.frombuffer(text, np.uint8).copy() if len(text) else np.zeros(1, np.uint8)
    seq = np.zeros((max(cap, 1), stride), np.uint8); qual = np.zeros((max(cap, 1), stride), np.uint8)
    ln = np.zeros(max(cap, 1), np.uint16); recs = np.zeros(max(cap, 1), capi.FASTQ_REC_DTYPE)
    info = capi.FastqInfo()
    rc = lib.fp_oracle_fastq_decode(buf.ctypes.data, len(text), final, phred64, stride, seq.ctypes.data, qual.ctypes.data, ln.ctypes.data, cap,
                                    recs.ctypes.data, C.byref(info))
    assert rc == 0
    n = int(info.n_records)
    return {"seq": seq[:n], "qual": qual[:n], "len": ln[:n], "recs": recs[:n], "info": info_dict(info)}


def oracle_fastq_encode(text, recs, res, seq, qual, stride):
    lib = oracle(); _bind_fastq(lib)
    n = len(recs)
    buf = np.frombuffer(text, np.uint8).copy() if len(text) else np.zeros(1, np.uint8)
    recs = np.ascontiguousarray(recs); res = np.ascontiguousarray(res); seq = np.ascontiguousarray(seq); qual = np.ascontiguousarray(qual)
    total = lib.fp_oracle_fastq_encode(buf.ctypes.data, recs.ctypes.data, res.ctypes.data, seq.ctypes.data, qual.ctypes.data, stride, n, None, 0)
    out = np.zeros(max(int(total), 1), np.uint8)
    got = lib.fp_oracle_fastq_encode(buf.ctypes.data, recs.ctypes.data, res.ctypes.data, seq.ctypes.data, qual.ctypes.data, stride, n, out.ctypes.data, int(total))
    assert got == total
    return out[:total].tobytes()


def ref_fastq_read(path, phred64=0):
    """The reference's FastqReader over a file: list of (name, seq, strand, qual) byte strings."""
    lib = ref()
    lib.fp_ref_fastq_read_file.restype = C.c_int64
    lib.fp_ref_fastq_read_file.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    cap = os.path.getsize(path) * 2 + 4096
    out = np.zeros(cap, np.uint8); used = C.c_int64()
    n = lib.fp_ref_fastq_read_file(str(path).encode(), phred64, out.ctypes.data, cap, C.byref(used))
    assert used.value <= cap
    recs, o = [], 0
    for _ in range(n):
        h = out[o:o + 16].view(np.int32); o += 16
        f = []
        for k in range(4):
            f.append(out[o:o + int(h[k])].tobytes()); o += int(h[k])
        recs.append(tuple(f))
    return recs


def decoded_fields(text, d):
    """(name, seq, strand, qual) tuples of a decode result, for comparison with ref_fastq_read."""
    out = []
    for i in range(len(d["recs"])):
        r = d["recs"][i]; n = int(d["len"][i])
        out.append((text[int(r["name_off"]):int(r["name_off"]) + int(r["name_len"])], d["seq"][i, :n].tobytes(),
                    text[int(r["strand_off"]):int(r["strand_off"]) + int(r["strand_len"])], d["qual"][i, :n].tobytes()))
    return out


def fastq_edge_cases():
    """name -> text: the line / record rules of FastqReader::getLine and ::read, one quirk each."""
    rec = lambda i, s, q, nm="r", st="+": f"@{nm}{i}\n{s}\n{st}\n{q}\n"        # noqa: E731
    good = "".join(rec(i, "ACGTN" * (i % 7 + 1), "IIII#" * (i % 7 + 1)) for i in range(40))
    return {
        "plain": good.encode(),
        "crlf": good.replace("\n", "\r\n").encode(),
        "lone_cr": good.replace("\n", "\r").encode(),
        "mixed_eol": (rec(0, "ACGT", "IIII") + rec(1, "ACG", "III").replace("\n", "\r\n") + rec(2, "AC", "II").replace("\n", "\r") + rec(3, "A", "I")).encode(),
        "no_final_newline": good.rstrip("\n").encode(),
        "blank_lines_between": ("\n\n" + rec(0, "ACGT", "IIII") + "\n" + rec(1, "GG", "##") + "\n\n\n" + rec(2, "TTT", "ABC")).encode(),
        "junk_before_name": ("garbage line\nmore junk\n" + rec(0, "ACGT", "IIII") + "not a name\n" + rec(1, "GG", "##")).encode(),
        "quality_starts_with_at": (rec(0, "ACGT", "@III") + rec(1, "GGTT", "@@@@") + rec(2, "AC", "+I")).encode(),
        "plus_with_name": "".join(rec(i, "ACGTAC", "IIIIII", st=f"+r{i}") for i in range(5)).encode(),
        "empty_reads": (rec(0, "", "") + rec(1, "ACGT", "IIII") + rec(2, "", "")).encode(),
        "bad_strand": (rec(0, "ACGT", "IIII") + rec(1, "ACGT", "IIII") + "@r2\nACGT\n-\nIIII\n" + rec(3, "ACGT", "IIII")).encode(),
        "empty_strand": (rec(0, "ACGT", "IIII") + "@r1\nACGT\n\nIIII\n" + rec(2, "ACGT", "IIII")).encode(),
        "length_mismatch": (rec(0, "ACGT", "IIII") + "@r1\nACGT\n+\nIII\n" + rec(2, "ACGT", "IIII")).encode(),
        "truncated_record": (good + "@last\nACGT\n+\n").encode(),
        "only_newlines": b"\n\n\n",
        "empty": b"",
        "long_names": "".join(rec(i, "ACGTACGTAC", "IIIIIIIIII", nm="instrument:run:flowcell:lane:tile:" + "x" * 300 + ":") for i in range(9)).encode(),
        "name_only_at": "@\nAC\n+\nII\n".encode(),
    }


def fastq_fuzz_text(rng, nrec=30):
    """Random FASTQ-ish text: mixed line ends, blank / junk lines between records, odd strand lines, empty reads,
    occasional broken records, optional missing final terminator."""
    eols = ["\n", "\r\n", "\r"]
    out = []
    for i in range(nrec):
        e = eols[int(rng.integers(0, 3))] if rng.random() < 0.3 else "\n"
        if rng.random() < 0.15:
            out.append(["", "junk", "+", "#comment", "\t"][int(rng.integers(0, 5))] + e)
        n = int(rng.integers(0, 40))
        s = "".join(rng.choice(list("ACGTN"), n)) if n else ""
        q = "".join(chr(int(x)) for x in rng.integers(33, 75, n)) if n else ""
        if n and rng.random() < 0.1:
            q = "@" + q[1:]
        strand = "+" if rng.random() < 0.8 else "+" + "x" * int(rng.integers(1, 9))
        r = rng.random()
        if r < 0.02:
            strand = "-"                               # reader stops here
        elif r < 0.04:
            q = q + "I"                                # length mismatch: reader stops here
        out.append(f"@r{i} {'y' * int(rng.integers(0, 20))}{e}{s}{e}{strand}{e}{q}{e}")
    text = "".join(out)
    if rng.random() < 0.3 and text:
        text = text.rstrip("\r\n")
    return text.encode()


def random_params(rng, paired, lib=None):
    """A random but valid option set: every knob the chain reads gets exercised in combinations no fixed config has."""
    R = lambda a, b: int(rng.integers(a, b + 1))          # noqa: E731
    coin = lambda p=0.5: bool(rng.random() < p)           # noqa: E731
    kw = dict(
        thread0_semantics=1 if coin(0.8) else 0,
        trim_front1=R(0, 8) if coin(0.4) else 0, trim_tail1=R(0, 8) if coin(0.4) else 0,
        max_len1=R(60, 140) if coin(0.3) else 0,
        cut_front=int(coin(0.4)), cut_tail=int(coin(0.4)), cut_right=int(coin(0.5)),
        cut_front_window=R(1, 8), cut_front_quality=R(5, 30), cut_tail_window=R(1, 8), cut_tail_quality=R(5, 30),
        cut_right_window=4 if coin(0.5) else R(1, 10), cut_right_quality=R(10, 30),
        polyg_enabled=int(coin()), polyg_min_len=R(5, 20), polyx_enabled=int(coin()), polyx_min_len=R(5, 20),
        adapter_enabled=int(coin(0.85)), dimer_max_len=R(0, 12),
        qual_filter_enabled=int(coin(0.85)), qualified_qual=33 + R(5, 30), unqualified_percent_limit=R(5, 80),
        n_base_limit=R(0, 10), avg_qual_req=R(0, 30) if coin(0.4) else 0,
        length_filter_enabled=int(coin(0.85)), length_required=R(0, 80), length_limit=R(100, 150) if coin(0.3) else 0,
        complexity_filter_enabled=int(coin(0.4)), complexity_threshold=R(5, 60) / 100.0,
    )
    if coin(0.5):
        kw["adapter_seq_r1"] = TRUSEQ_R1[: R(6, len(TRUSEQ_R1))]
    if coin(0.3):
        kw["fasta_adapters"] = [TRUSEQ_R1[: R(8, 33)], "CTGTCTCTTATACACATCT", "G" * R(8, 14)][: R(1, 3)]
    if paired:
        kw.update(trim_front2=R(0, 8) if coin(0.4) else 0, trim_tail2=R(0, 8) if coin(0.4) else 0, max_len2=R(60, 140) if coin(0.3) else 0,
                  correction_enabled=int(coin()), overlap_require=R(10, 40), overlap_diff_limit=R(1, 8), overlap_diff_percent_limit=R(5, 40),
                  allow_gap_overlap_trimming=int(coin(0.3)), insert_size_max=R(300, 600) if coin(0.3) else 512)
        if coin(0.5):
            kw["adapter_seq_r2"] = TRUSEQ_R2[: R(6, len(TRUSEQ_R2))]
        if coin(0.25):                                    # merging mode (drawn last: the earlier knobs keep their streams)
            kw.update(merge_enabled=1, merge_include_unmerged=int(coin()))
    return capi.default_params(paired, lib=lib or oracle(), **kw), kw


# ---------------- adapter-string histograms (SURVEY 8f rank 3) ----------------
MAX_ADAPTER_REC, LOW_COMPLEXITY_SKIP = 20000, 5000          # src/filterresult.cpp:7-8


def _low_complexity(a):                                    # FilterResult::isLowComplexity src/filterresult.cpp:116-123
    return sum(1 for i in range(len(a) - 1) if a[i] != a[i + 1]) < len(a) // 2


def rebuild_adapter_maps(events, arrs, adapters):
    """What the reference-side shim does with the device's fp_adapter_event list: sort by (unit, key) and replay
    FilterResult::addAdapterTrimmed (src/filterresult.cpp:124-180) in input order, with its caps and its early return.
    arrs = the rows AFTER the pass (corrected bytes); adapters = [adapter_seq_r1, adapter_seq_r2, fasta...]."""
    maps = ({}, {})

    def add(m, s):          # returns False when the reference `return`s out of the whole call
        if s in m:
            m[s] += 1
            return True
        if len(m) > MAX_ADAPTER_REC or (len(m) > LOW_COMPLEXITY_SKIP and _low_complexity(s)):
            return False
        m[s] = 1
        return True

    def text(e):
        if e["kind"] == 2:
            return adapters[e["adapter"]][: e["len"]]
        row = arrs["seq2" if e["which"] else "seq1"][e["unit"]]
        return bytes(row[e["start"]: e["start"] + e["len"]]).decode()
    ev = np.sort(events, order=["unit", "key"])
    i = 0
    while i < len(ev):
        e = ev[i]
        if e["kind"] == 0:                                   # addAdapterTrimmed(adapter1, adapter2): two events of one unit
            e2 = ev[i + 1]
            assert e2["kind"] == 0 and e2["unit"] == e["unit"] and e["which"] == 0 and e2["which"] == 1
            a1, a2 = text(e), text(e2)
            ok = True
            if a1:
                ok = add(maps[0], a1)
            if ok and a2:                                    # an early return on adapter1 skips adapter2 (SURVEY App. A.7)
                add(maps[1], a2)
            i += 2
        else:
            s = text(e)
            if s:
                add(maps[1] if e["which"] else maps[0], s)
            i += 1
    return maps


def ref_adapter_maps(params, arrs, cycles):
    """The reference's own mAdapter1 / mAdapter2 after a single-worker pass (oracle/_ref)."""
    a = {k: v.copy() for k, v in arrs.items()}
    b = capi.batch_from_arrays(a)
    paired = bool(params.paired)
    L = capi.make_layout(oracle(), paired, cycles, params.insert_size_max, params=params)
    cnt = np.zeros(L.total, np.int64)
    out = C.create_string_buffer(1 << 26); used = C.c_int64()
    r = ref()
    r.fp_ref_process_maps.restype = C.c_int
    r.fp_ref_process_maps.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.CounterLayout), C.POINTER(capi.Batch), C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    r.fp_ref_process_maps(C.byref(params), C.byref(L), C.byref(b), cnt.ctypes.data, out, len(out), C.byref(used))
    maps = ({}, {})
    for line in out.raw[:used.value].decode().splitlines():
        w, s, c = line.split("\t")
        maps[int(w) - 1][s] = int(c)
    return maps, capi.CounterView(L, cnt)
