"""Flower level, no GPU: the golden fixture is what the UNMODIFIED reference library produces here (when oracle/_ref holds
it), the harness's canonical post-bar() dump does not depend on the OpenMP team size, and the generators are deterministic."""
import numpy as np
import pytest

import _flowers as F
import _flower_golden as G


def test_fixture_has_the_references_own_flower():
    names = [c[0] for c in G.cases()]
    assert "shared_maxlen2" in names and "shared_iterator" in names and len(names) >= 10
    for name, fl, params, stream, bar in G.cases():
        assert stream[0] > 0 and bar[0] > 0, name


def test_random_flower_is_deterministic():
    a, b = F.random_flower(3), F.random_flower(3)
    assert a["seqs"] == b["seqs"] and a["adj"] == b["adj"]


@pytest.mark.skipif(not F.have("ref"), reason="oracle/_ref/libflower_ref.so not built (needs the reference's sources, see oracle/Makefile)")
def test_reference_library_reproduces_the_fixture():
    for name, fl, params, stream, bar in G.cases():
        r = F.blocks("ref", fl, params)
        assert np.array_equal(r["raw"], stream), name
    some = [c for c in G.cases() if c[0].startswith("random_")]
    out = F.bar("ref", [c[1] for c in some], threads=3)          # several flowers in ONE bar() call, three threads
    for c, o in zip(some, out):
        assert np.array_equal(o, c[4]), c[0]


@pytest.mark.skipif(not F.have("standin"), reason="oracle/_ref/libflower_standin.so not built (needs the reference's sources, see oracle/Makefile)")
def test_shims_and_host_code_over_a_standin_device_reproduce_the_fixture():
    """no GPU: the REAL shims (shim/cactus_bar_shim.c incl. its bar()) and the REAL host code of the product (host_bar.cpp,
    end_queue.h, bar_windows.h) under the reference's own flower-level objects, with a TEST-ONLY CPU stand-in for the device
    layer (tests/hosttest/standin_device.cpp: every job computed by the host build of the product's graph code). The GPU
    suite runs the same checks against the real libbarb200 (tests/test_gpu_flowers.py)."""
    for name, fl, params, stream, bar in G.cases():
        r = F.blocks("standin", fl, params)
        assert np.array_equal(r["raw"], stream), name
        assert np.array_equal(F.bar("standin", [fl], params)[0], bar), name
    flowers = [F.random_flower(100 + s, n_threads=int(4 + s % 5), n_blocks=int(2 + s % 4), seg_len=40 + 7 * (s % 9)) for s in range(24)]
    got = F.bar("standin", flowers, threads=4)                    # 24 flowers in one bar() call: submit all, then collect
    want = F.bar("ref", flowers, threads=2)
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), i


@pytest.mark.skipif(not (F.have("harvest") and F.have("standin")), reason="oracle/_ref/libflower_harvest.so not built (needs the reference's sources, see oracle/Makefile)")
def test_harvested_inputs_replay_to_the_same_alignments(tmp_path, oracle_built):
    """shim/cactus_bar_harvest.c records the inputs of every top-level alignment call of a REFERENCE bar() run (the way real
    datasets are to be captured for bench.py --workload); replaying the record through the product's host code (stand-in
    device) and through the oracle gives the same MSAs"""
    import os
    import workload
    import _reflib as R
    dump = str(tmp_path / "bar.harvest")
    flowers = [F.random_flower(300 + s, n_threads=5, n_blocks=3, seg_len=50) for s in range(5)]
    os.environ["BARB200_HARVEST"] = dump
    try:
        got = F.bar("harvest", flowers, threads=2)
    finally:
        del os.environ["BARB200_HARVEST"]
    want = F.bar("ref", flowers, threads=2)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)                     # recording does not change the run
    recs = workload.read_harvest(dump)
    assert len(recs) == len(flowers)
    assert sorted(sum(len(e) for e in r["ends"]) for r in recs) == sorted(2 * len(f["adj"]) for f in flowers)
    multi = [r for r in recs if r["right_end_indexes"] is not None]
    res, rcs, _ = R.hosttest_flowers([(r["ends"], r["right_end_indexes"], r["right_end_row_indexes"], r["overlaps"]) for r in multi])
    assert not rcs.any()
    for r, ms in zip(multi, res):
        o = R.oracle_make_consistent_partial_order_alignments(r["ends"], r["right_end_indexes"], r["right_end_row_indexes"], r["overlaps"])
        for a, b in zip(ms, o):
            assert a.shape == b.shape and np.array_equal(a, b)


PECAN = {"bar/partialOrderAlignment": "0"}


def pecan_flowers():
    """ends with up to 8 strings (all-pairs path of makeAlignment) and with 14+ strings (the incremental pair selection,
    multipleAligner.c:887-939: spanningTrees * (n - 1) < n (n - 1) / 2)"""
    return [F.random_flower(400 + s, n_threads=int(5 + s % 4), n_blocks=3, seg_len=60) for s in range(3)] + \
           [F.random_flower(500 + s, n_threads=14 + s, n_blocks=2, seg_len=70, p_skip=0.0, p_loop=0.0) for s in range(2)]


@pytest.mark.skipif(not F.have("standin"), reason="oracle/_ref/libflower_standin.so not built (needs the reference's sources, see oracle/Makefile)")
def test_cpecan_configuration_through_the_pecan_shim_on_the_standin_device():
    """bar() with partialOrderAlignment="0": the reference's makeFlowerAlignment3 / makeEndAlignment / poset code over
    shim/cactus_pecan_shim.c (makeAlignment with every selection round as one device batch, makeAllPairwiseAlignments,
    getAlignedPairsUsingAnchors). One OpenMP thread: the reference's tie breaks draw from ONE st_random() stream, so its own
    output depends on the thread interleaving."""
    fls = pecan_flowers()
    want = F.bar("ref", fls, PECAN, threads=1)
    got = F.bar("standin", fls, PECAN, threads=1)
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), i
