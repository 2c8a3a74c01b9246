"""FASTQ text <-> rows (SURVEY 8f rank 1): the CPU restatement of FastqReader::getLine/read and Read::appendToString
(oracle/fastp_oracle.c) pinned against the reference's own FastqReader (oracle/_ref, built from src/fastqreader.cpp),
plus size-independent properties of the codec.  The -m gpu twin (tests/test_gpu_fastq.py) holds the CUDA path to this oracle."""
import numpy as np
import pytest

import fp_testlib as T
from fastp_b200 import capi

CASES = T.fastq_edge_cases()


def ref_fastq_read_text(tmp_path, text, phred64=0):
    path = tmp_path / "in.fq"
    path.write_bytes(text)
    return T.ref_fastq_read(path, phred64)


@pytest.mark.reference
@pytest.mark.parametrize("name", list(CASES))
def test_oracle_decode_matches_fastqreader(tmp_path, name):
    text = CASES[name]
    d = T.oracle_fastq_decode(text, final=1, stride=512)
    got = T.decoded_fields(text, d)
    T.check_reference(f"fastq_decode/{name}", got, lambda: ref_fastq_read_text(tmp_path, text))
    if name in ("bad_strand", "empty_strand"):
        assert d["info"]["error"] == 1 and d["info"]["error_record"] == len(got)
    elif name == "length_mismatch":
        assert d["info"]["error"] == 2 and d["info"]["error_record"] == 1
    else:
        assert d["info"]["error"] == 0 and d["info"]["error_record"] == -1


@pytest.mark.reference
def test_oracle_decode_phred64_matches_fastqreader(tmp_path):
    rng = np.random.default_rng(3)
    recs = []
    for i in range(50):
        n = int(rng.integers(1, 60))
        s = "".join(rng.choice(list("ACGTN"), n)); q = bytes(rng.integers(59, 127, n).astype(np.uint8)).decode("latin1")
        recs.append(f"@p{i}\n{s}\n+\n{q}\n")
    text = "".join(recs).encode("latin1")
    d = T.oracle_fastq_decode(text, final=1, phred64=1, stride=64)
    T.check_reference("fastq_decode_phred64", T.decoded_fields(text, d), lambda: ref_fastq_read_text(tmp_path, text, phred64=1))


@pytest.mark.parametrize("name", ["plain", "crlf", "blank_lines_between", "junk_before_name", "quality_starts_with_at", "long_names", "truncated_record"])
@pytest.mark.parametrize("cut", [1, 7, 64, 1000])
def test_chunked_decode_equals_whole(name, cut):
    """Streaming contract: decode a chunk, carry the unconsumed tail into the next chunk -- same records as one call."""
    text = CASES[name]
    whole = T.decoded_fields(text, T.oracle_fastq_decode(text, final=1, stride=512))
    got, carry, pos = [], b"", 0
    while True:
        piece = text[pos:pos + cut]; pos += cut
        final = 1 if pos >= len(text) else 0
        chunk = carry + piece
        d = T.oracle_fastq_decode(chunk, final=final, stride=512)
        got += T.decoded_fields(chunk, d)
        carry = chunk[d["info"]["consumed"]:]
        if final:
            break
    assert got == whole


def test_encode_of_untouched_reads_is_the_canonical_text():
    text = CASES["crlf"]
    d = T.oracle_fastq_decode(text, final=1, stride=64)
    n = len(d["recs"])
    res = np.zeros(n, capi.READ_RESULT_DTYPE)
    res["len"] = d["len"]
    out = T.oracle_fastq_encode(text, d["recs"], res, d["seq"], d["qual"], 64)
    assert out == CASES["plain"]                       # same records, '\n' line ends (Read::appendToString always writes '\n')
    res["pair_verdict"][::2] = 3                       # failed reads are not written
    res["front"][1::2] = 1; res["len"][1::2] -= 2      # trimmed window
    out = T.oracle_fastq_encode(text, d["recs"], res, d["seq"], d["qual"], 64)
    lines = CASES["plain"].decode().split("\n")
    want = "".join(f"{lines[4 * i]}\n{lines[4 * i + 1][1:-1]}\n+\n{lines[4 * i + 3][1:-1]}\n" for i in range(1, n, 2))
    assert out.decode() == want


def test_capacity_limit_reports_more():
    text = CASES["plain"]
    d = T.oracle_fastq_decode(text, final=1, stride=64, capacity=5)
    assert d["info"]["n_records"] == 5 and d["info"]["more"] == 1
    rest = text[d["info"]["consumed"]:]
    d2 = T.oracle_fastq_decode(rest, final=1, stride=64)
    assert d["info"]["n_records"] + d2["info"]["n_records"] == 40


@pytest.mark.reference
def test_oracle_decode_fuzz_matches_fastqreader(tmp_path):
    """300 random texts (mixed line ends, junk, broken records): same records as the reference's FastqReader."""
    rng = np.random.default_rng(2026)
    for k in range(300):
        text = T.fastq_fuzz_text(rng)
        got = T.decoded_fields(text, T.oracle_fastq_decode(text, final=1, stride=64))
        T.check_reference(f"fastq_fuzz/{k}", got, lambda: ref_fastq_read_text(tmp_path, text))


@pytest.mark.reference
@pytest.mark.parametrize("paired", [1, 0])
@pytest.mark.parametrize("case", ["default", "full"])
def test_oracle_text_pipeline_equals_reference_cli(tmp_path, case, paired):
    """decode -> operator chain -> encode, all in the C port, against the UNMODIFIED reference CLI's output files: pins the whole
    text-path oracle (the -m gpu twin holds fp_fastq_process_host to the same files)."""
    import test_gpu_fastq as G
    flags, p, t1, t2 = G.cli_inputs(case, paired, n=2000)
    d1 = T.oracle_fastq_decode(t1, stride=160)
    arrs = {"seq1": d1["seq"].copy(), "qual1": d1["qual"].copy(), "len1": d1["len"].copy()}
    if paired:
        d2 = T.oracle_fastq_decode(t2, stride=160)
        arrs.update(seq2=d2["seq"].copy(), qual2=d2["qual"].copy(), len2=d2["len"].copy())
    res = T.run_cpu("oracle", p, arrs, 160)
    got = [T.oracle_fastq_encode(t1, d1["recs"], res["out1"], res["arrs"]["seq1"], res["arrs"]["qual1"], 160)]
    if paired:
        got.append(T.oracle_fastq_encode(t2, d2["recs"], res["out2"], res["arrs"]["seq2"], res["arrs"]["qual2"], 160))
    T.check_reference(f"cli_text/{case}/{paired}", got, lambda: G.run_cli(tmp_path, flags, t1, t2))
