"""cPecan mode, CPU suite: (1) the plain-C oracle against the compiled reference (differential, seeded) and against the
committed golden vectors, incl. the reference's own known-answer case; (2) the product's block program
(cactus_b200/csrc/pecan_cta.cuh) and host planning (pecan_plan.cpp), emulated on the host by tests/hosttest, against the
oracle -- bit-exact on the integer triples AND on the pre-floor posteriors; (3) the host-only C-ABI helpers
(barb200_pecan_band / barb200_pecan_split_points) against the oracle. The CUDA kernel itself runs under -m gpu."""
import numpy as np
import pytest

import _golden as G
import _reflib as R
from _synth import pecan_pair
import workload  # noqa: E402


def _params(c):
    return R.pecan_params(threshold=c["threshold"], min_diags=c["min_diags"], tb_diags=c["tb_diags"], expansion=c["expansion"])


def _random_case(rng):
    L = int(rng.choice([1, 7, 30, 100, 300, 600, 1500]))
    sx, sy, a = pecan_pair(rng, L, k_anchor=int(rng.choice([8, 12, 20])), keep=float(rng.choice([1, 0.7, 0.3, 0.0])),
                           sub=float(rng.choice([0.02, 0.1, 0.3])), ins=float(rng.choice([0.0, 0.01, 0.05])),
                           dele=float(rng.choice([0.0, 0.01, 0.05])), nfrac=float(rng.choice([0, 0, 0.03])))
    rl, rr = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
    sb = int(rng.choice([30 * 30, 100 * 100, 400 * 400, 3000 * 3000]))
    p = R.pecan_params(threshold=float(rng.choice([0.01, 0.2, 0.0001, 0.0])), min_diags=int(rng.choice([1000, 100, 50])),
                       tb_diags=int(rng.choice([40, 10, 1])), expansion=int(rng.choice([20, 4, 10, 0])))
    return sx, sy, a, rl, rr, p, sb


def test_oracle_golden(oracle_built):
    n = 0
    for c in G.pecan_cases():
        t, po = R.oracle_pecan_aligned_pairs(c["sx"], c["sy"], c["anchors"], c["rl"], c["rr"], _params(c), c["split"])
        assert np.array_equal(t, c["triples"]), c["id"]
        if "post" in c:
            x, y, ps = R.oracle_pecan_posteriors(c["sx"], c["sy"], c["anchors"], c["rl"], c["rr"], _params(c))
            assert np.array_equal(x, c["post_x"]) and np.array_equal(y, c["post_y"]) and np.array_equal(ps, c["post"]), c["id"]
        n += 1
    assert n >= 10


def test_reference_known_answer(oracle_built):
    """submodules/cPecan/tests/pairwiseAlignerTest.c:243-322: AGCG vs AGTTCG, threshold 0.2 -> exactly these four pairs"""
    c = next(G.pecan_cases())
    assert (c["sx"], c["sy"]) == (b"AGCG", b"AGTTCG")
    want = {(0, 0), (1, 1), (2, 4), (3, 5)}
    assert {(int(x), int(y)) for _, x, y in c["triples"]} == want
    t, _, _ = R.hosttest_pecan_aligned_pairs(c["sx"], c["sy"], c["anchors"], c["rl"], c["rr"], _params(c), c["split"])
    assert {(int(x), int(y)) for _, x, y in t} == want


def random_reference_cases():
    """the seeded cases of test_oracle_vs_reference_random: (key, inputs digest, case, whether the posteriors of its single
    sub-matrix are compared too)"""
    rng = np.random.default_rng(4242)
    for it in range(60):
        sx, sy, a, rl, rr, p, sb = _random_case(rng)
        inputs = G.digest(np.frombuffer(sx, np.uint8), np.frombuffer(sy, np.uint8), np.asarray(a, np.int64).reshape(-1, 2),
                          np.array([rl, rr, sb], np.int64), np.frombuffer(bytes(p), np.uint8))
        single = len(R.oracle_pecan_split_points(len(sx), len(sy), a, sb, rl, rr)) == 1
        yield "pecan_random/%d" % it, inputs, (sx, sy, a, rl, rr, p, sb), single


def test_oracle_vs_reference_random(oracle_built):
    """the oracle's triples (and, for a single sub-matrix, its pre-floor posteriors) against the unmodified reference's, stored as
    digests in tests/golden/ref_digests.json (scripts/make_golden_ref_digests.py)"""
    for key, inputs, (sx, sy, a, rl, rr, p, sb), single in random_reference_cases():
        out = {"triples": G.digest(R.oracle_pecan_aligned_pairs(sx, sy, a, rl, rr, p, sb)[0])}
        if single:
            out["posteriors"] = G.digest(*R.oracle_pecan_posteriors(sx, sy, a, rl, rr, p))
        G.check_ref_digest(key, inputs, out)


def test_warp_program_golden():
    for c in G.pecan_cases():
        t, po, cells = R.hosttest_pecan_aligned_pairs(c["sx"], c["sy"], c["anchors"], c["rl"], c["rr"], _params(c), c["split"])
        assert np.array_equal(t, c["triples"]), c["id"]
        if "post" in c:
            assert np.array_equal(po[::-1], c["post"]), c["id"]      # the public call returns a region's pairs reversed


def test_warp_program_vs_oracle_random(oracle_built):
    rng = np.random.default_rng(777)
    for it in range(80):
        sx, sy, a, rl, rr, p, sb = _random_case(rng)
        to, po = R.oracle_pecan_aligned_pairs(sx, sy, a, rl, rr, p, sb)
        T = int(rng.choice([32, 128, 256]))
        th, ph, cells = R.hosttest_pecan_aligned_pairs(sx, sy, a, rl, rr, p, sb, threads=T, ring_width=int(rng.choice([0, 8, 40, 96, 608])),
                                                       ring_extra=int(rng.choice([0, 0, 7, 300])))
        assert np.array_equal(to, th) and np.array_equal(po, ph), (it, T, len(sx), len(sy), len(a))


def test_empty_and_degenerate(oracle_built):
    p = R.pecan_params()
    for sx, sy in [(b"", b""), (b"A", b""), (b"", b"ACGT"), (b"A", b"A"), (b"NNNN", b"NNNN"), (b"acgt", b"ACGT")]:
        to, po = R.oracle_pecan_aligned_pairs(sx, sy, [], False, False, p)
        th, ph, _ = R.hosttest_pecan_aligned_pairs(sx, sy, [], False, False, p)
        assert np.array_equal(to, th) and np.array_equal(po, ph), (sx, sy)


def test_cabi_band_and_split_points(oracle_built):
    """host-only entry points of libbarb200.so (no GPU needed)"""
    import cactus_b200 as cb
    from cactus_b200 import build as b
    b.build()
    rng = np.random.default_rng(99)
    for it in range(40):
        sx, sy, a, rl, rr, p, sb = _random_case(rng)
        L, Rr = cb.pecan_band(len(sx), len(sy), a, int(p.diagonalExpansion))
        Lo, Ro = R.oracle_pecan_band(len(sx), len(sy), a, int(p.diagonalExpansion))
        assert np.array_equal(L, Lo) and np.array_equal(Rr, Ro), it
        sp = cb.pecan_split_points(len(sx), len(sy), a, sb, rl, rr)
        assert np.array_equal(sp, R.oracle_pecan_split_points(len(sx), len(sy), a, sb, rl, rr)), it
    with pytest.raises(cb.BarB200Error):
        cb.pecan_band(10, 10, [[5, 5], [4, 6]], 20)         # anchors must increase (the reference asserts)


def test_block_program_bench_shape(oracle_built):
    """the benchmark's pair shape (2 kbp, anchors = exact runs >= 50 bp) in the kernel's production configuration:
    128 threads per block, 320 ring positions in the shared part, the flanks of the wide diagonals in the overflow block"""
    import cactus_b200 as cb
    from cactus_b200 import build as b
    b.build()
    for sx, sy, a, _, _ in workload.synth_pairs(7, 2, 2000, k_anchor=50):
        to, po = R.oracle_pecan_aligned_pairs(sx, sy, a, False, False, R.pecan_params())
        th, ph, cells = R.hosttest_pecan_aligned_pairs(sx, sy, a, False, False, R.pecan_params(), threads=128, ring_width=320)
        assert np.array_equal(to, th) and np.array_equal(po, ph)
        L, Rr = cb.pecan_band(len(sx), len(sy), a, 20)
        assert cells == int(((Rr - L) // 2 + 1).sum()) and ((Rr - L) // 2 + 1).max() > 320      # wide enough to use the overflow


def test_reference_invariants_on_the_block_program():
    """the reference's own validity checks (submodules/cPecan/tests/pairwiseAlignerTest.c:345-382 checkAlignedPairs, used by
    test_getAlignedPairsWithBanding :404-450 on random sequences of length 0..100 and their evolved copies): scores in
    (0, PAIR_ALIGNMENT_PROB_1], coordinates inside the sequences, every (x, y) reported once"""
    from _synth import evolve, to_ascii
    rng = np.random.default_rng(404)
    for it in range(60):
        L = int(rng.integers(0, 101))
        x = rng.integers(0, 4, L).astype(np.uint8)
        sx = to_ascii(x) if L else b""
        sy = to_ascii(evolve(x, rng, sub=0.1, ins=0.05, dele=0.05)) if L else b""
        t, po, cells = R.hosttest_pecan_aligned_pairs(sx, sy, [], bool(it & 1), bool(it & 2), R.pecan_params(), threads=int(rng.choice([32, 128])))
        if len(t) == 0:
            continue
        assert t[:, 0].min() > 0 and t[:, 0].max() <= 10000000
        assert t[:, 1].min() >= 0 and t[:, 1].max() < len(sx) and t[:, 2].min() >= 0 and t[:, 2].max() < len(sy)
        assert len({(int(a), int(b)) for _, a, b in t}) == len(t)
        assert cells == (len(sx) + 1) * (len(sy) + 1)          # no anchors: the band is the whole matrix
