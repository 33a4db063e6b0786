"""Readers for the committed golden vectors (tests/golden/*.npz, produced from the unmodified reference by
scripts/make_golden.py) and for the reference's output digests of the seeded differential tests (tests/golden/ref_digests.json,
scripts/make_golden_ref_digests.py)."""
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF_DIGESTS = os.path.join(GOLD, "ref_digests.json")


def digest(*arrays):
    """sha256 (first 16 hex digits) over the dtype, shape and bytes of each array"""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(repr((a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()[:16]


def trace_digest(tr):
    """the fields of an _reflib trace that the differential tests compare, reduced to digests and scalars"""
    alns = tr["alns"]
    return {"msa_len": int(tr["msa_len"]), "cells": int(tr["cells"]), "msa": digest(tr["msa"]),
            "order": digest(np.array(tr["read_id_map"], np.int64)),
            "alns": digest(np.array([[a["read_id"], a["qlen"], a["node_n"], a["best_score"]] for a in alns], np.int64).reshape(-1, 4)),
            "cigar": digest(*[a["cigar"] for a in alns]),
            "dp": digest(*[np.concatenate([a["dp_beg"], a["dp_end"]]) for a in alns])}


_ref_digests = None


def check_ref_digest(key, inputs, out):
    """`out` (a dict of digests and scalars) must equal what the unmodified reference produced for the case `key`, whose
    inputs had the digest `inputs`"""
    global _ref_digests
    if _ref_digests is None:
        with open(REF_DIGESTS) as f:
            _ref_digests = json.load(f)
    want = _ref_digests[key]
    assert inputs == want["in"], "%s: the inputs are not the ones the reference's digests were made from" % key
    diff = {k: (out.get(k), want["out"].get(k)) for k in set(out) | set(want["out"]) if out.get(k) != want["out"].get(k)}
    assert not diff, "%s differs from the reference (got, want): %s" % (key, diff)


def poa_cases():
    z = np.load(os.path.join(GOLD, "poa_golden.npz"))
    for ci in range(int(z["n_cases"][0])):
        lens = z[f"c{ci}_lens"]
        flat = z[f"c{ci}_flat"]
        offs = np.concatenate([[0], np.cumsum(lens)])
        seqs = [flat[offs[i]:offs[i + 1]] for i in range(len(lens))]
        pr = z[f"c{ci}_params"]
        params = dict(wb=int(pr[0]), wf=float(z[f"c{ci}_wf"][0]), o1=int(pr[1]), e1=int(pr[2]), o2=int(pr[3]),
                      e2=int(pr[4]), k=int(pr[5]), w=int(pr[6]), min_w=int(pr[7]), progressive=int(pr[8]),
                      disable_seeding=int(pr[9]))
        yield dict(id=ci, seqs=seqs, params=params, msa=z[f"c{ci}_msa"], order=[int(x) for x in z[f"c{ci}_order"]],
                   best=z[f"c{ci}_best"], ncigar=z[f"c{ci}_ncigar"], cigar=z[f"c{ci}_cigar"], beg=z[f"c{ci}_beg"],
                   end=z[f"c{ci}_end"], cells=int(z[f"c{ci}_cells"][0]))


def window_cases():
    z = np.load(os.path.join(GOLD, "bar_golden.npz"))
    for n in range(int(z["n_windows"][0])):
        strs = z[f"w{n}_strs"].tobytes().split(b"\n")
        yield dict(id=n, strs=strs, win=int(z[f"w{n}_win"][0]), msa=z[f"w{n}_msa"])


def two_end_cases():
    z = np.load(os.path.join(GOLD, "bar_golden.npz"))
    for m in range(int(z["n_two_end"][0])):
        ends = [z[f"t{m}_strs{e}"].tobytes().split(b"\n") for e in range(2)]
        rr = [[int(x) for x in z[f"t{m}_rr{e}"]] for e in range(2)]
        K = len(ends[0])
        yield dict(id=m, ends=ends, ri=[[1] * K, [0] * K], rr=rr,
                   ov=[[len(s) for s in ends[0]], [len(s) for s in ends[1]]], win=int(z[f"t{m}_win"][0]),
                   msas=[z[f"t{m}_msa{e}"] for e in range(2)])


def pecan_cases():
    """outputs of the reference's getAlignedPairsUsingAnchors / getPosteriorProbsWithBanding (scripts/make_golden_pecan.py);
    case 0 is the reference's own known-answer input (submodules/cPecan/tests/pairwiseAlignerTest.c:243-322)"""
    z = np.load(os.path.join(GOLD, "pecan_golden.npz"))
    for ci in range(int(z["n_cases"][0])):
        fl = z[f"c{ci}_flags"]
        c = dict(id=ci, sx=z[f"c{ci}_sx"].tobytes(), sy=z[f"c{ci}_sy"].tobytes(), anchors=z[f"c{ci}_anchors"],
                 rl=bool(fl[0]), rr=bool(fl[1]), min_diags=int(fl[2]), tb_diags=int(fl[3]), expansion=int(fl[4]),
                 split=int(fl[5]), threshold=float(z[f"c{ci}_thr"][0]), triples=z[f"c{ci}_triples"])
        if f"c{ci}_post" in z:
            c.update(post_x=z[f"c{ci}_post_x"], post_y=z[f"c{ci}_post_y"], post=z[f"c{ci}_post"])
        yield c
