"""Pin the plain-C oracle (oracle/poa_oracle.c, bar_oracle.c) against the UNMODIFIED reference: MSA bytes, guide-tree order,
every graph cigar, every dp_beg/dp_end, best scores and the banded cell count must be identical. The reference's outputs for
these seeded inputs are stored as digests in tests/golden/ref_digests.json (scripts/make_golden_ref_digests.py runs the
reference over the same case lists). CPU only."""
import numpy as np
import pytest

import _golden as G
import _reflib as R
from _synth import family, gapped_family, to_ascii, two_end_problem

GAP_MODELS = [(400, 30, 1200, 1), (4, 2, 24, 1), (400, 30, 1200, 30), (1200, 1, 400, 30), (400, 30, 300, 1), (6, 2, 6, 2)]


def assert_same_trace(a, b, tag):
    assert a["msa_len"] == b["msa_len"], tag
    assert np.array_equal(a["msa"], b["msa"]), tag
    assert a["read_id_map"] == b["read_id_map"], tag
    assert a["cells"] == b["cells"], tag
    for x, y in zip(a["alns"], b["alns"]):
        for k in ("read_id", "qlen", "node_n", "best_score"):
            assert x[k] == y[k], (tag, k)
        assert np.array_equal(x["cigar"], y["cigar"]), tag
        assert np.array_equal(x["dp_beg"], y["dp_beg"]), tag
        assert np.array_equal(x["dp_end"], y["dp_end"]), tag


def poa_inputs(seqs, p):
    return G.digest(*seqs, np.frombuffer(bytes(p), np.uint8))


def random_family_cases(seed):
    rng = np.random.default_rng(100 + seed)
    for it in range(12):
        K = int(rng.integers(2, 12))
        L = int(rng.choice([5, 20, 60, 150, 300, 400, 800]))
        kw = dict(sub=float(rng.choice([0.0, 0.02, 0.08, 0.2])), ins=float(rng.choice([0, 0.005, 0.03])),
                  dele=float(rng.choice([0, 0.005, 0.03])), nfrac=float(rng.choice([0, 0, 0.01])))
        seqs = family(rng, K, L, sort=bool(rng.random() < 0.7), **kw)
        p = R.cactus_params() if rng.random() < 0.6 else R.cactus_params(
            wb=int(rng.choice([10, 30, 100])), wf=float(rng.choice([0.01, 0.02, 0.1])), progressive=int(rng.integers(0, 2)))
        yield "poa_random_families/%d/%d" % (seed, it), seqs, p


def gap_model_cases(gaps):
    o1, e1, o2, e2 = gaps
    rng = np.random.default_rng(4242 + o1 + 7 * e2)
    p = R.cactus_params(o1=o1, e1=e1, o2=o2, e2=e2, wb=300, wf=0.05)
    for it in range(14):
        seqs = gapped_family(rng, int(rng.integers(3, 9)), int(rng.choice([120, 500, 1100])), [1, 2, 3, 8, 27, 28, 29, 33, 64, 65, 150, 300])
        yield "poa_gap_models/%d,%d,%d,%d/%d" % (o1, e1, o2, e2, it), seqs, p


def unrelated_ragged_cases():
    rng = np.random.default_rng(11)
    for it in range(60):
        K = int(rng.integers(2, 40))
        seqs = [rng.integers(0, 5 if rng.random() < 0.2 else 4, int(rng.integers(1, 500))).astype(np.uint8) for _ in range(K)]
        if rng.random() < 0.7:
            seqs.sort(key=lambda s: -len(s))
        p = R.cactus_params(wb=int(rng.choice([0, 1, 5, 10, 1000])), wf=float(rng.choice([0.0, 0.01, 0.1])),
                            progressive=int(rng.integers(0, 2)))
        yield "poa_unrelated_ragged/%d" % it, seqs, p


def bench_shape_cases():
    yield "poa_bench_shape", family(np.random.default_rng(3), 8, 2000), R.cactus_params()


def long_window_cases():
    seqs = family(np.random.default_rng(4), 4, 10000, sub=0.03, ins=0.01, dele=0.01)
    yield "poa_long_window", [s[:10000] for s in seqs], R.cactus_params()


def window_cases():
    rng = np.random.default_rng(5)
    for it in range(40):
        K = int(rng.integers(1, 8))
        L = int(rng.choice([10, 50, 200, 700]))
        strs = [to_ascii(s) for s in family(rng, K, L, sub=0.05, ins=0.02, dele=0.02, nfrac=0.01)]
        if rng.random() < 0.2 and K > 1:
            strs[-1] = b""
        win = int(rng.choice([5, 20, 50, 110, 10000]))
        yield "bar_windows/%d" % it, strs, win


def window_inputs(strs, win):
    return G.digest(np.frombuffer(b"\n".join(strs), np.uint8), np.array([len(strs), win], np.int64))


def two_end_cases():
    rng = np.random.default_rng(6)
    for it in range(20):
        K = int(rng.integers(1, 10))
        L = int(rng.choice([10, 60, 150]))
        ends, ri, rr, ov = two_end_problem(rng, K, L, sub=0.05, ins=0.02, dele=0.02)
        win = int(rng.choice([20, 10000]))
        yield "bar_two_ends/%d" % it, (ends, ri, rr, ov), win


def two_end_inputs(problem, win):
    ends, ri, rr, ov = problem
    return G.digest(*[np.frombuffer(b"\n".join(e), np.uint8) for e in ends], np.array(ri + rr + ov, np.int64), np.array([win], np.int64))


def msas_digest(msas):
    return {"shapes": [list(m.shape) for m in msas], "msas": G.digest(*msas)}


def check_trace(key, seqs, p, tr):
    G.check_ref_digest(key, poa_inputs(seqs, p), G.trace_digest(tr))


@pytest.mark.parametrize("seed", range(6))
def test_poa_msa_trace_random_families(oracle_built, seed):
    for key, seqs, p in random_family_cases(seed):
        check_trace(key, seqs, p, R.oracle_poa_msa_trace(seqs, p))


@pytest.mark.parametrize("gaps", GAP_MODELS)
def test_poa_msa_long_gaps_and_gap_models(oracle_built, gaps):
    """the inputs of test_gpu_parity.py::test_long_gaps_and_gap_models: the oracle (and the serial traceback the host build runs)
    against the reference, so that the GPU test's checker is pinned in these regimes too"""
    for it, (key, seqs, p) in enumerate(gap_model_cases(gaps)):
        check_trace(key, seqs, p, R.oracle_poa_msa_trace(seqs, p))
        if it < 4:
            check_trace(key, seqs, p, R.hosttest_poa_msa_trace(seqs, p))


def test_poa_msa_unrelated_ragged(oracle_built):
    """unrelated sequences, ragged lengths (1..500), N-rich, degenerate bands -- exercises the int16/int32 lane
    switch (abpoa_align_simd.c:1293-1302) and the adaptive band edges"""
    for key, seqs, p in unrelated_ragged_cases():
        check_trace(key, seqs, p, R.oracle_poa_msa_trace(seqs, p))


def test_poa_msa_bench_shape(oracle_built):
    """one end of the benchmark shape: 8 x 2 kbp, Cactus defaults (int32 lanes, band 1000+0.1L)"""
    for key, seqs, p in bench_shape_cases():
        check_trace(key, seqs, p, R.oracle_poa_msa_trace(seqs, p))


def test_poa_msa_long_window(oracle_built):
    """a full 10 kbp window (the largest DP the shim ever issues, cactus_progressive_config.xml:308)"""
    for key, seqs, p in long_window_cases():
        check_trace(key, seqs, p, R.oracle_poa_msa_trace(seqs, p))


def test_msa_make_partial_order_alignment_windows(oracle_built):
    """sliding windows + overlap trimming (poaBarAligner.c:463-749), incl. the empty-row N hack"""
    for key, strs, win in window_cases():
        b = R.oracle_msa_make_partial_order_alignment(strs, window_size=win)
        G.check_ref_digest(key, window_inputs(strs, win), msas_digest([b]))


def test_make_consistent_two_ends(oracle_built):
    """cross-end consistency trimming (poaBarAligner.c:751-801) on the reference's own two-end construction"""
    for key, problem, win in two_end_cases():
        ends, ri, rr, ov = problem
        b = R.oracle_make_consistent_partial_order_alignments(ends, ri, rr, ov, window_size=win)
        G.check_ref_digest(key, two_end_inputs(problem, win), msas_digest(b))
        # the reference's invariant (poaBarTest.c:160-176): kept prefix lengths of a shared string add up to its length
        for i in range(len(ends[0])):
            k = rr[0][i]
            kept1 = int((b[0][i] != 5).sum())
            kept2 = int((b[1][k] != 5).sum())
            assert kept1 + kept2 == len(ends[0][i])
