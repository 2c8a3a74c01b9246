"""Pins the plain-C port (oracle/fastp_oracle.c) against the REFERENCE's own objects compiled into
oracle/_ref/libfastp_ref.so (recipe: oracle/Makefile) on seeded synthetic batches: every per-read record,
overlap record, corrected base and counter, for every option set the parity tests use.
Where oracle/_ref is absent the reference's answers come from tests/golden/reference_digests.json (fp_testlib.check_reference)."""
import pytest

import fp_testlib as T

pytestmark = pytest.mark.reference


@pytest.mark.parametrize("paired", [1, 0])
@pytest.mark.parametrize("name", T.CONFIG_NAMES)
def test_port_equals_reference_objects(name, paired):
    p = T.config_params(name, paired)
    n = 4000 if name == "fasta_adapters" else 12000
    _, arrs = T.synth_host(n, 160, paired, 5000, 2024, 1, 150)
    x = T.run_cpu("oracle", p, arrs, 160)
    T.check_result_reference(f"objects/{name}/{paired}", x, p, arrs, 160, skip=("adapter_pos",))


@pytest.mark.parametrize("L,stride", [(150, 160), (100, 112), (250, 256)])
@pytest.mark.parametrize("name", T.GAP_CONFIG_NAMES)
def test_port_equals_reference_gap_overlap(name, L, stride):
    """--allow_gap_overlap_trimming: OverlapAnalysis::analyze(..., allowGap=true) + Matcher::diffWithOneInsertion
    (src/overlapanalysis.cpp:106-160, src/matcher.cpp:40-91) on reads that carry single-base indels."""
    p = T.config_params(name, 1)
    _, arrs = T.synth_host(8000, stride, 1, 300, 31, 2, L)
    x = T.run_cpu("oracle", p, arrs, stride)
    T.check_result_reference(f"gap/{name}/{L}", x, p, arrs, stride, skip=("adapter_pos",))


@pytest.mark.parametrize("L,stride", [(150, 160), (100, 112)])
@pytest.mark.parametrize("name", T.MERGE_CONFIG_NAMES)
def test_port_equals_reference_merge_mode(name, L, stride):
    """--merge / --include_unmerged (src/peprocessor.cpp:519-560, OverlapAnalysis::merge src/overlapanalysis.cpp:148-179): the second
    overlap analysis on the trimmed reads, the merged read's verdict (weight 2), post-filter Stats of read 1 over merged reads up to two
    rows long (counter block sized 2 x stride), mMergedPairs."""
    p = T.config_params(name, 1)
    _, arrs = T.synth_host(8000, stride, 1, 700, 77, 1, L)
    x = T.run_cpu("oracle", p, arrs, 2 * stride)
    T.check_result_reference(f"merge/{name}/{L}", x, p, arrs, 2 * stride, skip=("adapter_pos",))
    assert int(x["counters"].filter[107]) > 0, "no pair merged"


@pytest.mark.parametrize("L,stride", [(250, 256), (100, 112), (36, 48)])
def test_port_equals_reference_other_lengths(L, stride):
    p = T.config_params("cfg4_full", 1)
    _, arrs = T.synth_host(5000, stride, 1, 0, 7, 1, L)
    T.check_result_reference(f"lengths/{L}", T.run_cpu("oracle", p, arrs, stride), p, arrs, stride, skip=("adapter_pos",))


def test_reference_mt_equals_single_thread():
    """Stats::merge / FilterResult::merge are plain sums: the multi-threaded CPU baseline must give the same block as one thread
    (both pinned to the C port's answer on the same batch)."""
    p = T.config_params("cfg4_full", 1)
    _, arrs = T.synth_host(6000, 160, 1, 0, 11, 1, 150)
    x = T.run_cpu("oracle", p, arrs, 160)
    T.check_result_reference("mt/1", x, p, arrs, 160, skip=("adapter_pos",))
    T.check_result_reference("mt/5", x, p, arrs, 160, skip=("adapter_pos",), nthreads=5)


@pytest.mark.parametrize("paired", [1, 0])
@pytest.mark.parametrize("L,stride,sampling", [(150, 160, 20), (100, 112, 7), (250, 256, 3)])
def test_port_equals_reference_overrepresentation(paired, L, stride, sampling):
    """Stats::statRead's over-representation scan (stats.cpp:270-288) incl. the post-filter sampling by counted rank."""
    _, arrs = T.synth_host(6000, stride, paired, 0, 5, 1, L)
    p = T.overrep_params("cfg4_full", paired, arrs, L, sampling)
    x = T.run_cpu("oracle", p, arrs, stride)
    T.check_result_reference(f"overrep/{L}/{paired}", x, p, arrs, stride, skip=("adapter_pos",))
    assert sum(int(x["counters"].overrep(s)[0].sum()) for s in range(4 if paired else 2)) > 10


@pytest.mark.parametrize("paired", [1, 0])
def test_port_equals_reference_random_option_sets(paired):
    """30 random option sets (windows, thresholds, trims, adapter lists, overlap limits ...) on reads with indels."""
    import numpy as np
    rng = np.random.default_rng(1234 + paired)
    for k in range(30):
        p, kw = T.random_params(rng, paired)
        _, arrs = T.synth_host(1500, 160, paired, 100 * k, 900 + k, 2 if paired else 1, 150)
        x = T.run_cpu("oracle", p, arrs, 160)
        T.check_result_reference(f"random/{paired}/{k}", x, p, arrs, 160, skip=("adapter_pos",))
