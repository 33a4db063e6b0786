#!/usr/bin/env python
"""Generate tests/golden/ref_digests.json: the UNMODIFIED reference's outputs (oracle/_ref/*.so, built by oracle/Makefile from
the reference's sources) over the seeded case lists of tests/test_oracle_vs_ref.py and
tests/test_pecan_cpu.py::test_oracle_vs_reference_random, reduced to digests (tests/_golden.py), so that those tests compare
the oracle with the reference where the reference's sources are not available.

  python scripts/make_golden_ref_digests.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _golden as G  # noqa: E402
import _reflib as R  # noqa: E402
import test_oracle_vs_ref as T  # noqa: E402
import test_pecan_cpu as P  # noqa: E402


def main():
    assert R.have_ref() and R.have_bar_ref() and R.have_pecan_ref(), "build oracle/_ref first (make -C oracle ref)"
    out = {}
    poa = [c for s in range(6) for c in T.random_family_cases(s)] + [c for g in T.GAP_MODELS for c in T.gap_model_cases(g)] + \
        list(T.unrelated_ragged_cases()) + list(T.bench_shape_cases()) + list(T.long_window_cases())
    for key, seqs, p in poa:
        out[key] = {"in": T.poa_inputs(seqs, p), "out": G.trace_digest(R.ref_poa_msa_trace(seqs, p))}
    for key, strs, win in T.window_cases():
        out[key] = {"in": T.window_inputs(strs, win), "out": T.msas_digest([R.ref_msa_make_partial_order_alignment(strs, window_size=win)])}
    for key, problem, win in T.two_end_cases():
        out[key] = {"in": T.two_end_inputs(problem, win),
                    "out": T.msas_digest(R.ref_make_consistent_partial_order_alignments(*problem, window_size=win))}
    for key, inputs, (sx, sy, a, rl, rr, p, sb), single in P.random_reference_cases():
        o = {"triples": G.digest(R.ref_pecan_aligned_pairs(sx, sy, a, rl, rr, p, sb))}
        if single:
            o["posteriors"] = G.digest(*R.ref_pecan_posteriors(sx, sy, a, rl, rr, p))
        out[key] = {"in": inputs, "out": o}
    with open(G.REF_DIGESTS, "w") as f:
        f.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(v, sort_keys=True)) for k, v in out.items()) + "\n}\n")
    print(G.REF_DIGESTS, len(out), os.path.getsize(G.REF_DIGESTS))


if __name__ == "__main__":
    main()
