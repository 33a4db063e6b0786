#!/usr/bin/env python
"""bench.py -- BAR POA DP throughput (Gcell/s, ends/s) of the B200 engine vs the reference CPU BAR path.

Contract (see the round brief): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.
A *step* is one pass of the hot path (batched POA: all abpoa_msa jobs of a batch of ends) over one batch of synthetic
ends of BASELINE.json's shape: E ends x 8 sequences x 2 kbp per GPU (weak scaling; BASELINE.json configs[2] scaled to
what one step should take -- configs[1], evolverMammals, needs data that is not available offline).

  value   whole-job Gcell/s, inputs already resident in HBM (stage created before the timed region), device time of
          the kernel launches (CUDA events on the launching stream), max over ranks.
  e2e     the same metric through the C-ABI call a caller makes (barb200_poa_msa_batch) with HOST buffers: host
          packing + guide trees + H2D + kernel + D2H + unpack all inside the timed region.
  cells   the banded-cell definition of SURVEY.md 8d (sum of dp_end-dp_beg+1), counted by the kernel itself and
          pinned to the reference's count by the parity tests.

  parity  the GPU arm's in-run gate (BASELINE.md 3.5): the per-end MSA hashes of the CPU leg's sample must equal the GPU's; a
          mismatch aborts the run before any number is printed.
  shapes  device throughput of SURVEY.md 8d's scaled-down shapes and of one MIXED batch (bucketed by CTA class).
  e2e_flowers  flowers (4 ends each) driven through the end queue from 16 host threads: synchronous calls and submit-all /
          collect (barb200_flower_submit / _wait), next to the single-batch e2e.

`--impl reference` times the reference's own CPU implementation (unmodified abPOA built from /root/reference into
oracle/_ref, AVX2, OpenMP over ends with all host threads; the plain-C oracle port if that library is absent) on a
bounded sample of the same workload and prints the same line with "impl": "reference". That arm loads NO product code
(inputs come from workload/, a plain host library).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time


def _cpu_quota():
    """CPUs this container may really use: affinity mask capped by the cgroup quota (the GPU boxes show 128 logical CPUs under a 16-CPU quota)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:  # noqa: BLE001
        pass
    return n


# Thread pools sized for the 128 visible CPUs (numpy / torch / OpenMP defaults) spin on 128 threads under a 16-CPU quota and get the
# whole container throttled by the CFS bandwidth controller for hundreds of milliseconds at a time (seen as 250 ms stalls inside timed
# host-side calls; cpu.stat nr_throttled). Size them for the quota. Set before numpy / torch load. (OMP_WAIT_POLICY=passive on top of
# this cost the library's short parallel loops ~9 ms per step in wake-ups and is not needed once the pools fit the quota.)
for _k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
    os.environ.setdefault(_k, str(_cpu_quota()))

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import workload  # noqa: E402  (synthetic inputs: a plain host library shared by both arms, not product code)

K_SEQS, L_BP = 8, 2000
METRIC = "BAR POA DP Gcells/sec and ends/sec at 1/2/4/8 B200 vs reference CPU BAR"
ALGO_BYTES_PER_CELL = 32.0     # SURVEY.md 8d: 20 B written + 12 B read per cell (int32 planes)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled during the timed region. In-process NVML (nvidia_ml_py): spawning nvidia-smi five times a
    second takes the driver's global lock at every start and stalls the timed host-side CUDA calls (it cost the e2e leg ~20 ms of a
    260 ms step); the nvidia-smi query is the fallback when the module is missing."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []
        self.source = "nvml"
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:  # noqa: BLE001
            self.nv, self.h, self.source = None, None, "nvidia-smi"

    def _nvml_row(self):
        nv, h = self.nv, self.h
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:  # noqa: BLE001
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        bit = lambda name: "Active" if r & getattr(nv, name, 0) else "Not Active"   # noqa: E731
        return [str(sm), str(mx), "", hex(r), bit("nvmlClocksThrottleReasonHwSlowdown"), bit("nvmlClocksThrottleReasonHwThermalSlowdown"),
                bit("nvmlClocksThrottleReasonSwThermalSlowdown"), bit("nvmlClocksThrottleReasonSwPowerCap")]

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                if self.nv is not None:
                    self.rows.append(self._nvml_row())
                else:
                    o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                       capture_output=True, text=True, timeout=5).stdout.strip()
                    if o:
                        self.rows.append([x.strip() for x in o.split(",")])
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.1 if self.nv is not None else 1.0)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "source": self.source}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "samples": len(self.rows), "reasons": sorted(reasons), "source": self.source}


def usable_cores():
    """host threads the box really gives us (oversubscribing the quota makes the CPU arm slower, not faster)"""
    return _cpu_quota()


PECAN_BYTES_PER_CELL = 120.0   # SURVEY.md 8d: 5 fp64 states x (forward write + forward read at the traceback + backward write)

# --dump-outputs keeps every per-end / per-pair summary but the full alignments of a fixed sample only (64 MB in all at most)
DUMP_SAMPLE_ENDS, DUMP_SAMPLE_PAIRS = 256, 64


def _dump_sample(n, k):
    """a fixed, seeded choice of min(n, k) of n indices, increasing"""
    return np.sort(np.random.default_rng(0).choice(n, min(n, k), replace=False))


def dump_poa_outputs(d, msas, cells):
    """what the batched POA returned after the last timed step: every end's MSA width, banded cells and FNV-1a MSA hash (as
    its two 32-bit halves, exact in float64), and the MSA bytes of a fixed sample of ends (each [K, width] matrix flattened,
    concatenated in the order of poa_sample_ends)"""
    os.makedirs(d, exist_ok=True)
    idx = _dump_sample(len(msas), DUMP_SAMPLE_ENDS)
    h = np.array([workload.msa_hash(m) for m in msas], np.uint64)
    np.save(os.path.join(d, "poa_msa_columns.npy"), np.array([m.shape[1] for m in msas], np.float64))
    np.save(os.path.join(d, "poa_cells.npy"), np.asarray(cells, np.float64))
    np.save(os.path.join(d, "poa_msa_hash.npy"), np.stack([h >> np.uint64(32), h & np.uint64(0xffffffff)], 1).astype(np.float64))
    np.save(os.path.join(d, "poa_sample_ends.npy"), idx.astype(np.float64))
    np.save(os.path.join(d, "poa_sample_msa.npy"), np.concatenate([msas[i].reshape(-1) for i in idx]).astype(np.float32))


def dump_pecan_outputs(d, res):
    """what the pair-HMM stage returned after the last timed step: every pair's triple count, banded cells and sum of integer
    scores, and the (score, x, y) triples and pre-floor posteriors of a fixed sample of pairs (concatenated in the order of
    pecan_sample_pairs)"""
    os.makedirs(d, exist_ok=True)
    idx = _dump_sample(len(res), DUMP_SAMPLE_PAIRS)
    np.save(os.path.join(d, "pecan_triples_per_pair.npy"), np.array([len(r[0]) for r in res], np.float64))
    np.save(os.path.join(d, "pecan_cells.npy"), np.array([r[2] for r in res], np.float64))
    np.save(os.path.join(d, "pecan_score_sums.npy"), np.array([r[0][:, 0].sum() for r in res], np.float64))
    np.save(os.path.join(d, "pecan_sample_pairs.npy"), idx.astype(np.float64))
    np.save(os.path.join(d, "pecan_sample_triples.npy"), np.concatenate([res[i][0] for i in idx]).reshape(-1, 3).astype(np.float64))
    np.save(os.path.join(d, "pecan_sample_posteriors.npy"), np.concatenate([res[i][1] for i in idx]).astype(np.float64))


def pecan_measure(local_rank, rank, first_pair, n_pairs, steps, warmup, cpu_budget, want_cpu, no_e2e, host_threads, dump_dir=None):
    """cPecan mode (SURVEY.md 8a row a13, BASELINE.json configs[3]): banded pair-HMM posteriors of n_pairs synthetic
    2 kbp pairs per GPU per step with MUM-like anchors (k = 50, Cactus' setting). Runs in a process of its own (see main)
    and returns this rank's raw measurements."""
    import cactus_b200 as cb
    eng = cb.Engine(cb.PoaParams(device=local_rank, host_threads=host_threads))
    pairs = workload.synth_pairs(first_pair, n_pairs, L_BP, k_anchor=50)
    st = eng.pecan_stage(pairs)
    cells = float(st.cells())
    for _ in range(warmup):
        st.run()
    dev_ms, launches = 0.0, 0
    for _ in range(steps):
        dev_ms += st.run()             # CUDA-event time of the launch(es); the call returns after the stream is idle
        launches += st.launches()
    res = st.fetch(True)
    if dump_dir:
        dump_pecan_outputs(dump_dir, res)
    n_trip = int(sum(len(r[0]) for r in res))
    st.close()
    out = {"dev_ms": dev_ms, "launches": launches, "cells": cells, "n_pairs": n_pairs, "steps": steps, "e2e_ms": float("nan"), "same": True,
           "h2d": int(sum(len(q[0]) + len(q[1]) + q[2].nbytes for q in pairs)), "d2h": n_trip * 24}
    if not no_e2e:
        # the timed call is the C ABI itself (host strings + anchors in, malloc'd triples out); building the ctypes argument
        # arrays before and turning the outputs into numpy arrays after are harness work
        table = eng.pecan_table(pairs)
        eng._take_pairs(*eng.pecan_batch_raw(table), table.n)                  # warm-up (also sizes the context's caches)
        t0 = time.time()
        raw = eng.pecan_batch_raw(table)                                       # synchronous: returns with the results on the host
        out["e2e_ms"] = (time.time() - t0) * 1e3
        res2 = eng._take_pairs(*raw, table.n)
        out["same"] = bool(all(np.array_equal(a[0], b[0]) for a, b in zip(res, res2)))
    if want_cpu and rank == 0:
        try:
            import _reflib as R
            threads = usable_cores()
            samp = [(q[0], q[1], q[2], False, False) for q in pairs[: max(2, threads)]]
            s0, kind = R.cpu_pecan_many(samp, threads)
            n = int(min(n_pairs, max(len(samp), cpu_budget / max(s0 / len(samp), 1e-6))))
            samp = [(q[0], q[1], q[2], False, False) for q in pairs[:n]]
            secs, kind = R.cpu_pecan_many(samp, threads)
            c = float(sum(r[2] for r in res[:n]))
            # parity on the sample actually timed: the reference's triples must equal the engine's
            chk = R.ref_pecan_aligned_pairs(*samp[0], R.pecan_params()) if kind == "reference" else R.oracle_pecan_aligned_pairs(*samp[0], R.pecan_params())[0]
            out["cpu_baseline"] = {"value": c / secs / 1e9, "unit": "Gcell/s", "pairs_per_s": n / secs, "cores": threads, "kind": kind,
                                   "sample": "first %d of the step's pairs, %.1f s wall, one getAlignedPairsUsingAnchors call per pair on a pool of %d threads" % (n, secs, threads),
                                   "bit_identical_on_first_pair": bool(np.array_equal(chk, res[0][0]))}
            # SURVEY.md 8d: max abs difference of the pre-floor posteriors (tolerance 1e-5; the engine is held to 0) on a few pairs,
            # against the plain-C oracle (itself pinned bit for bit to the compiled reference by tests/test_pecan_cpu.py)
            md = 0.0
            for q, r in list(zip(samp, res))[:4]:
                to, po = R.oracle_pecan_aligned_pairs(q[0], q[1], q[2], False, False, R.pecan_params())
                md = max(md, float(np.max(np.abs(po - r[1]))) if len(po) == len(r[1]) and len(po) else (0.0 if len(po) == len(r[1]) else float("inf")))
            out["cpu_baseline"]["max_abs_posterior_diff_4_pairs"] = md
        except Exception as e:  # noqa: BLE001
            out["cpu_baseline"] = {"value": None, "unit": "Gcell/s", "cores": usable_cores(), "kind": "unavailable", "sample": str(e)}
    eng.close()
    return out


def reference_pecan(R, args, threads):
    """the reference's own getAlignedPairsUsingAnchors on the host cores, bounded sample of the cPecan workload; cells from the
    checker's band (sum of diagonal widths over the split regions), the same definition the engine reports"""
    pairs = workload.synth_pairs(0, min(args.pecan_pairs_per_step, 4 * max(2, threads) * (args.steps + args.warmup)), L_BP, k_anchor=50)
    samp = [(q[0], q[1], q[2], False, False) for q in pairs[: max(2, threads)]]
    s0, kind = R.cpu_pecan_many(samp, threads)
    n = int(min(len(pairs), max(len(samp), min(args.cpu_budget, 12.0) / max(s0 / len(samp), 1e-6) / max(1, args.steps + args.warmup))))
    samp = [(q[0], q[1], q[2], False, False) for q in pairs[:n]]

    def cells_of(q):
        c = 0
        sp = R.oracle_pecan_split_points(len(q[0]), len(q[1]), q[2], 3000 * 3000, False, False)
        j = 0
        for x1, y1, x2, y2 in sp:
            sub = []
            while j < len(q[2]) and q[2][j][0] + q[2][j][1] < x2 + y2:
                sub.append((q[2][j][0] - x1, q[2][j][1] - y1))
                j += 1
            L, Rr = R.oracle_pecan_band(int(x2 - x1), int(y2 - y1), np.array(sub, np.int64).reshape(-1, 2), 20)
            c += int(((Rr - L) // 2 + 1).sum())
        return c
    ncount = min(n, 8)
    cells_per_pair = sum(cells_of(q) for q in samp[:ncount]) / ncount
    for _ in range(args.warmup):
        R.cpu_pecan_many(samp, threads)
    t = 0.0
    for _ in range(args.steps):
        s, kind = R.cpu_pecan_many(samp, threads)
        t += s
    value = cells_per_pair * n * args.steps / t / 1e9
    return {"metric": "cPecan banded pair-HMM forward/backward/posterior Gcell/s (cells = sum of band diagonal widths)", "value": value, "unit": "Gcell/s",
            "impl": "reference", "pairs_per_s": n * args.steps / t, "ms_per_step": t / args.steps * 1e3, "dtype": "f64",
            "cpu_baseline": {"value": value, "unit": "Gcell/s", "cores": threads, "kind": kind,
                             "sample": "%d pairs (2 kbp, MUM-like anchors) per step, cells/pair from an exact count of %d pairs" % (n, ncount)}}


def pecan_object(mine, mx, sm, n_pairs):
    """the "pecan" object of the JSON line from rank 0's measurements (mine) and the reductions over ranks"""
    peak, peak_src = measured_peak()
    steps = mine["steps"]
    tot_cells, tot_pairs = float(sm[2]), float(sm[3])
    launch_ms = mine["dev_ms"] / max(1, mine["launches"])
    achieved = mine["cells"] * (steps / max(1, mine["launches"])) * PECAN_BYTES_PER_CELL / (launch_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json")))["pecan_dram_bytes_per_cell"] * mine["cells"] * (steps / max(1, mine["launches"]))
    except Exception:  # noqa: BLE001
        pass
    out = {"metric": "cPecan banded pair-HMM forward/backward/posterior Gcell/s (cells = sum of band diagonal widths)",
           "value": tot_cells * steps / float(mx[0]) / 1e6, "unit": "Gcell/s", "pairs_per_s": tot_pairs * steps / float(mx[0]) * 1e3,
           "ms_per_step": float(mx[0]) / steps, "dtype": "f64",
           "config": {"workload": "synthetic %d pairs x %d bp per GPU per step, 2%% sub / 0.5%% ins / 0.5%% del, anchors = exact co-linear "
                                  "runs >= 50 bp (MUM-like), diagonalExpansion 20, threshold 0.01" % (n_pairs, L_BP),
                      "cells_per_pair": mine["cells"] / n_pairs},
           "e2e": {"value": tot_cells / float(mx[1]) / 1e6, "unit": "Gcell/s", "pairs_per_s": tot_pairs / float(mx[1]) * 1e3, "ms_per_step": float(mx[1]),
                   "h2d_bytes_per_step": mine["h2d"], "d2h_bytes_per_step": mine["d2h"],
                   "api": "barb200_pecan_aligned_pairs_batch (host strings + anchors -> (score, x, y) triples)", "same_as_staged": bool(mine["same"])},
           "gpu_launches": int(sm[4]),
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                        "peak_source": peak_src, "kernel": "pecan_posterior_kernel", "bytes_per_cell_algorithmic": PECAN_BYTES_PER_CELL}}
    if "cpu_baseline" in mine:
        out["cpu_baseline"] = mine["cpu_baseline"]
    return out



def cpu_poa_leg(n_seq, lens, flat, threads, budget_s, min_ends):
    """The reference CPU path on the host cores over a bounded sample of the step's ends: OpenMP schedule(dynamic,1) over ends (the
    reference's own unit of parallelism, bar/impl/bar.c:90-94), at least `min_ends` ends so that every thread gets several.
    Timed twice: with glibc's default allocator and with large blocks retained (the stand-in for the jemalloc Cactus links,
    oracle/ref_harness.c: ref_malloc_mode). Returns (dict, n, hashes of the n ends)."""
    import _reflib as R
    K = K_SEQS
    offs = np.concatenate([[0], np.cumsum(lens)])
    n0 = int(min(len(n_seq), max(2, threads)))
    secs0, kind, _ = R.cpu_poa_msa_many(n_seq[:n0], lens[:n0 * K], flat[:offs[n0 * K]], threads=threads, malloc_mode=1)
    per_end = secs0 / n0
    n = int(min(len(n_seq), max(min_ends, n0, budget_s / 2 / max(per_end, 1e-6))))
    res = {}
    hashes = None
    for mode, name in ((0, "glibc_default"), (1, "retained_blocks")):
        secs, kind, _, h = R.cpu_poa_msa_many(n_seq[:n], lens[:n * K], flat[:offs[n * K]], threads=threads, malloc_mode=mode, want_hashes=True)
        res[name] = secs
        hashes = h
    return res, kind, n, hashes


def reference_arm(args):
    """`--impl reference`: the reference's CPU implementation of both sections, rank 0 only; no product library is loaded"""
    import ctypes as C
    import _reflib as R
    E = args.ends_per_step
    threads = usable_cores()
    K = K_SEQS
    # a bounded sample per step: at least 8 ends per thread, so that schedule(dynamic,1) keeps every core busy to the end
    n = int(min(E, max(8 * threads, 32)))
    n_seq, lens, flat = workload.synth_ends(0, n, K, L_BP)
    offs = np.concatenate([[0], np.cumsum(lens)])
    lib = R._load(R.build_oracle())
    lib.oracle_poa_cells.restype = C.c_int64
    lib.oracle_poa_cells.argtypes = [C.POINTER(R.RefParams), C.c_int, C.c_void_p, C.c_void_p]
    p = R.cactus_params()
    ncount = min(n, 4)                     # cells per end from an exact count of a few ends (all ends have the same shape)
    csum = 0
    for e in range(ncount):
        ln = np.ascontiguousarray(lens[e * K:(e + 1) * K])
        f = np.ascontiguousarray(flat[offs[e * K]:offs[(e + 1) * K]])
        csum += lib.oracle_poa_cells(C.byref(p), K, ln.ctypes.data, f.ctypes.data)
    cells_per_end = csum / ncount
    times = {}
    kind = "reference"
    for mode, name in ((0, "glibc_default"), (1, "retained_blocks")):
        for _ in range(args.warmup if mode == 1 else min(args.warmup, 1)):
            R.cpu_poa_msa_many(n_seq, lens, flat, threads=threads, malloc_mode=mode)
        t = 0.0
        k = args.steps if mode == 1 else 1
        for _ in range(k):
            s, kind, _ = R.cpu_poa_msa_many(n_seq, lens, flat, threads=threads, malloc_mode=mode)
            t += s
        times[name] = t / k
    best = min(times.values())
    value = cells_per_end * n / best / 1e9
    config = workload_config(E, 1)
    line = {"metric": METRIC, "value": value, "unit": "Gcell/s", "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": best * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config, "ends_per_s": n / best,
            "cpu_baseline": {"value": value, "unit": "Gcell/s", "cores": threads, "kind": kind,
                             "sample": "%d ends (8 x 2 kbp) per step (>= 8 per thread), OpenMP schedule(dynamic,1) over ends; cells/end from an exact count of %d ends" % (n, ncount),
                             "allocator": {"glibc_default_gcells": cells_per_end * n / times["glibc_default"] / 1e9,
                                           "retained_blocks_gcells": cells_per_end * n / times["retained_blocks"] / 1e9,
                                           "note": "Cactus links jemalloc (include.mk:53-64); its autoconf build cannot run here, so glibc is told to retain and reuse "
                                                   "large blocks instead (ref_malloc_mode); value = the faster of the two"},
                             "per_thread_gcells": value / threads},
            "e2e": {"value": value, "unit": "Gcell/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.pecan_pairs_per_step > 0:
        try:
            line["pecan"] = reference_pecan(R, args, threads)
        except Exception as e:  # noqa: BLE001
            line["pecan"] = {"error": str(e)}
    try:                # this arm must not map any product code (the judge checks the loaded libraries)
        line["product_library_loaded"] = "libbarb200" in open("/proc/self/maps").read()
    except Exception:  # noqa: BLE001
        pass
    print(json.dumps(line))
    return 0


def workload_config(E, world):
    return {"workload": "synthetic %d ends x %d seqs x %d bp per GPU per step, Cactus default POA parameters "
                        "(convex gap 400/30/1200/1, band 1000+0.1L, progressive order), 2%% sub / 0.5%% ins / 0.5%% del" % (E, K_SEQS, L_BP),
            "ends_per_gpu_per_step": E, "seqs_per_end": K_SEQS, "bp": L_BP, "parallelism": "ends sharded over %d GPU(s)" % world,
            "l2": "working set (DP planes, ~40 MB per resident CTA) is far larger than the 126 MB L2"}


SHAPES = [("1000x8x200", 1000, 8, 200), ("1000x4x2000", 1000, 4, 2000), ("100x30x2000", 100, 30, 2000), ("10x8x10000", 10, 8, 10000)]
MIXED = [(2000, 8, 200), (300, 8, 2000), (8, 8, 10000)]


def shapes_leg(eng):
    """device throughput of SURVEY.md 8d's scaled-down shapes, of one end-level shape with several windows (10 x 8 x 25 kbp, through the
    end queue) and of one MIXED batch next to its three parts run alone (the buckets share the GPU; N1 of the round-1 verdict)"""
    out = {}

    def run_stage(packed, reps=2):
        st = eng.stage(packed=packed)
        st.run()
        ms = min(st.run() for _ in range(reps))
        _, cells = st.fetch()
        b = st.buckets()
        st.close()
        return ms, float(cells.sum()), b
    for name, n, k, l in SHAPES:
        ms, cells, b = run_stage(workload.synth_ends(7000000, n, k, l))
        out[name] = {"gcells_per_s": cells / ms / 1e6, "ends_per_s": n / ms * 1e3, "ms": ms, "buckets": b}
    # 10 ends x 8 x 25 kbp: five windows per end, through msa_make_partial_order_alignment (host strings, wall clock)
    n_seq, lens, flat = workload.synth_ends(7100000, 10, 8, 25000)
    offs = np.concatenate([[0], np.cumsum(lens)])
    asc = np.frombuffer(b"ACGTN", np.uint8)
    ends = [[asc[flat[offs[e * 8 + i]:offs[e * 8 + i + 1]]].tobytes() for i in range(8)] for e in range(10)]
    eng.msa_make_partial_order_alignment_batch(ends[:2])
    t0 = time.time()
    ms_ = eng.msa_make_partial_order_alignment_batch(ends)
    dt = time.time() - t0
    out["10x8x25000"] = {"ends_per_s": 10 / dt, "ms": dt * 1e3, "columns": int(np.mean([m.column_no for m in ms_])),
                         "api": "barb200_msa_make_partial_order_alignment_batch (host strings, 5 windows per end, wall clock)"}
    parts, alone = [], 0.0
    for i, (n, k, l) in enumerate(MIXED):
        pk = workload.synth_ends(7200000 + 100000 * i, n, k, l)
        ms, cells, _ = run_stage(pk)
        alone += ms
        parts.append(pk)
    mixed = (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]), np.concatenate([p[2] for p in parts]))
    ms, cells, b = run_stage(mixed)
    out["mixed"] = {"what": " + ".join("%d x (%d, %d)" % m for m in MIXED), "gcells_per_s": cells / ms / 1e6, "ms": ms, "sum_of_parts_alone_ms": alone,
                    "ratio_to_sum_of_parts": ms / alone, "buckets": b}
    return out


def flowers_leg(eng, first_flower, n_flowers, threads, cells_per_end, flowers=None):
    """N synthetic flowers (4 ends x 8 x 2 kbp each, ends pairwise reverse complements: cross-end trimming does real work) through the
    end queue from `threads` host threads: (a) synchronous barb200_make_consistent_partial_order_alignments calls, (b) every thread
    submits its flowers (barb200_flower_submit) before it collects them (barb200_flower_wait) -- what the shim's bar() does.
    The ctypes argument tables are built before the clock starts; Msa -> numpy conversion is not part of the timed calls."""
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor
    from cactus_b200.api import _StrTable
    if flowers is None:
        flowers = workload.synth_flowers(first_flower, n_flowers, 4, K_SEQS, L_BP)
    n_flowers = len(flowers)
    lib, ctx = eng.lib, eng.ctx

    def tables(fl):
        ends, ri, rr, ov = fl[:4]
        t = _StrTable(ends)
        keep = []

        def tab(rows):
            if rows is None:
                return None
            arr = (C.c_void_p * len(rows))()
            for i, r in enumerate(rows):
                a = (C.c_int64 * len(r))(*[int(v) for v in r])
                keep.append(a)
                arr[i] = C.cast(a, C.c_void_p)
            return arr
        return (t, tab(ri), tab(rr), tab(ov), keep, len(ends))
    tabs = [tables(f) for f in flowers]

    def free_msas(ms, n):
        for i in range(n):
            lib.barb200_msa_destruct(ms[i])
        lib.barb200_free(C.cast(ms, C.c_void_p))

    def sync_worker(tid):
        for f in range(tid, n_flowers, threads):
            t, ri, rr, ov, _, n = tabs[f]
            if ri is not None:
                ms = lib.barb200_make_consistent_partial_order_alignments(ctx, n, t.seq_no, t.strs, t.lens, ri, rr, ov, 10000, 5000, 1.0)
            else:                                       # a single-end record: the synchronous call is submit + wait
                h = lib.barb200_flower_submit(ctx, n, t.seq_no, t.strs, t.lens, None, None, None, 10000, 5000, 1.0)
                ms = lib.barb200_flower_wait(ctx, h) if h else None
            if not ms:
                raise RuntimeError(lib.barb200_last_error(ctx).decode())
            free_msas(ms, n)

    def async_worker(tid):
        mine = list(range(tid, n_flowers, threads))
        tickets = []
        for f in mine:
            t, ri, rr, ov, _, n = tabs[f]
            h = lib.barb200_flower_submit(ctx, n, t.seq_no, t.strs, t.lens, ri, rr, ov, 10000, 5000, 1.0)
            if not h:
                raise RuntimeError(lib.barb200_last_error(ctx).decode())
            tickets.append(h)
        for f, h in zip(mine, tickets):
            ms = lib.barb200_flower_wait(ctx, h)
            if not ms:
                raise RuntimeError(lib.barb200_last_error(ctx).decode())
            free_msas(ms, tabs[f][5])
    res = {}
    n_ends_total = sum(len(f[0]) for f in flowers)
    cells = cells_per_end * n_ends_total
    for name, worker in (("sync_calls", sync_worker), ("submit_all_then_collect", async_worker)):
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(worker, range(threads)))          # warm-up (sizes the lanes' arenas)
        q0 = eng.queue_stats()
        t0 = time.time()
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(worker, range(threads)))
        dt = time.time() - t0
        q1 = eng.queue_stats()
        res[name] = {"gcells_per_s": cells / dt / 1e9, "ends_per_s": n_ends_total / dt, "ms": dt * 1e3, "device_batches": q1["batches"] - q0["batches"]}
    res["flowers"] = n_flowers
    res["ends"] = n_ends_total
    res["host_threads"] = threads
    return res, flowers


def replay_arm(args):
    """`--workload <file>`: the BAR inputs of a real run recorded by shim/cactus_bar_harvest.c (workload.read_harvest), replayed through
    the end queue from 16 host threads (synchronous calls and submit-all / collect), next to the reference library on a bounded
    sample of the same flowers, with the MSAs of that sample compared byte for byte. ends/s and bases/s (no cell count: the
    flower-level API does not return one)."""
    import cactus_b200 as cb
    import _reflib as R
    recs = workload.read_harvest(args.workload)
    flowers = [(r["ends"], r["right_end_indexes"], r["right_end_row_indexes"], r["overlaps"]) for r in recs]
    windows = sorted({(r["window_size"], r["max_prog_rows"], r["max_prog_length_diff"]) for r in recs})
    if len(windows) != 1 or windows[0] != (10000, 5000, 1.0):
        sys.stderr.write("[bench] note: the record uses window / progressive parameters %s; the replay uses Cactus' defaults\n" % (windows,))
    bases = sum(len(s) for f in flowers for e in f[0] for s in e)
    eng = cb.Engine(cb.PoaParams(host_threads=usable_cores()))
    res, _ = flowers_leg(eng, 0, len(flowers), 16, 0.0, flowers=flowers)
    for k in ("sync_calls", "submit_all_then_collect"):
        res[k]["bases_per_s"] = bases / (res[k]["ms"] * 1e-3)
        del res[k]["gcells_per_s"]
    # reference library on a bounded sample + parity of that sample
    sample = [f for f in flowers if f[1] is not None][: max(1, min(len(flowers), 4 * usable_cores()))]
    t0 = time.time()
    same = True
    for f in sample:
        want = R.ref_make_consistent_partial_order_alignments(f[0], f[1], f[2], f[3])
        got = eng.make_consistent_partial_order_alignments(f[0], f[1], f[2], f[3])
        same = same and all(a.msa_seq.shape == b.shape and np.array_equal(a.msa_seq, b) for a, b in zip(got, want))
    line = {"metric": "BAR POA ends/s on harvested inputs (replay of %s)" % os.path.basename(args.workload), "unit": "ends/s",
            "value": res["submit_all_then_collect"]["ends_per_s"], "n_gpus": 1, "data": "harvested", "higher_is_better": True,
            "config": {"workload": "replay of %d recorded flowers, %d ends, %d bases" % (len(flowers), res["ends"], bases)},
            "replay": res, "parity": {"flowers_checked": len(sample), "identical": bool(same), "seconds_incl_reference": time.time() - t0}}
    eng.close()
    if not same:
        sys.stderr.write("[bench] PARITY GATE FAILED on the replayed sample\n")
        return 3
    print(json.dumps(line))
    return 0


def gpu_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    # host threads per rank: the box's usable cores shared by the ranks of this node, but never fewer than 8 (the host side of a
    # batch is bursty: the ranks' bursts rarely coincide). torchrun exports OMP_NUM_THREADS=1, hence the explicit value.
    cores = usable_cores()
    host_threads = max(1, min(cores, max(8, (2 * cores) // local_world))) if local_world > 1 else cores
    E = args.ends_per_step
    config = workload_config(E, world)
    import cactus_b200 as cb
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        saved = os.dup(1)
        os.dup2(2, 1)              # NCCL prints its version banner on stdout at the first collective; the JSON line must stand alone
        try:
            dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    dev = torch.device("cuda", local_rank)

    # rank 0 deals the end list out (scatter) -- the only exchange the path needs before the compute
    from cactus_b200 import dist as D
    ranges = D.deal_end_ranges(E * world, world) if rank == 0 else None
    first_end, n_ends = D.scatter_end_ranges(ranges, dev) if world > 1 else (0, E)

    eng = cb.Engine(cb.PoaParams(device=local_rank, host_threads=host_threads))
    n_seq, lens, flat = workload.synth_ends(first_end, n_ends, K_SEQS, L_BP)
    stage = eng.stage(packed=(n_seq, lens, flat))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        stage.run()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    t0 = time.time()
    dev_ms = 0.0
    launches = 0
    for _ in range(args.steps):
        dev_ms += stage.run()          # CUDA-event time of the launch(es) on the launching stream
        launches += stage.launches()
    barrier()
    wall_ms = (time.time() - t0) * 1e3
    msas, cells = stage.fetch()
    if args.dump_outputs and rank == 0:
        dump_poa_outputs(args.dump_outputs, msas, cells)
    my_cells = float(cells.sum())
    buckets = stage.buckets()

    # ---- e2e through the host-buffer C-ABI call ----
    # inputs in PINNED host memory; per step: pack + guide trees + H2D + kernels + D2H + unpack (all inside
    # barb200_poa_msa_batch), and for N > 1 the gather of every rank's MSA bytes on rank 0 over NCCL (send / recv of the
    # un-padded bytes into one device buffer, one copy into pinned host memory): alignments come back to the process that owns
    # the flowers.
    import ctypes as C
    pin = [torch.from_numpy(a).pin_memory() for a in (n_seq, lens, flat)]
    p_nseq, p_lens, p_flat = [t.numpy() for t in pin]
    phases = {"build_ms": 0.0, "run_ms": 0.0, "device_ms": 0.0, "fetch_ms": 0.0, "total_ms": 0.0, "gather_ms": 0.0, "calls": 0}

    def e2e_once():
        outs = (C.c_void_p * n_ends)()
        ml = np.zeros(n_ends, np.int32)
        cc = np.zeros(n_ends, np.int64)
        eng._check(eng.lib.barb200_poa_msa_batch(eng.ctx, n_ends, p_nseq.ctypes.data, p_lens.ctypes.data, p_flat.ctypes.data, None,
                                                 outs, ml.ctypes.data, cc.ctypes.data))
        tm = eng.last_batch_timing()
        for k in ("build_ms", "run_ms", "device_ms", "fetch_ms", "total_ms"):
            phases[k] += tm[k]
        phases["calls"] += 1
        d2h = int((ml.astype(np.int64) * K_SEQS).sum())
        if world > 1:
            tg = time.time()
            D.gather_msa_bytes(outs, ml, K_SEQS, dev)
            phases["gather_ms"] += (time.time() - tg) * 1e3
        eng.lib.barb200_free_many(outs, n_ends)
        return d2h
    d2h, e2e_ms = 0, float("nan")
    if not args.no_e2e:
        e2e_once()
        for k in phases:
            phases[k] = 0.0
        barrier()
        t1 = time.time()
        for _ in range(args.steps):
            d2h = e2e_once()
        barrier()
        e2e_ms = (time.time() - t1) * 1e3 / args.steps
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- reduce over ranks: max time, sum cells; gather alignment checksums on rank 0 ----
    mx, sm = D.reduce_stats([dev_ms, wall_ms, e2e_ms, my_cells, float(n_ends), float(launches)], dev)
    checksums = D.gather_checksums(float(sum(int(m.sum()) for m in msas[:64])), dev)

    # ---- rank 0 only from here on (the other ranks wait at the barrier before the cPecan section) ----
    extra = {}
    if rank == 0:
        # parity gate + CPU baseline: the reference on the host cores over a bounded sample of the step's ends
        if not args.no_cpu_baseline:
            try:
                secs, kind, n_cpu, hashes = cpu_poa_leg(n_seq, lens, flat, cores, args.cpu_budget, 8 * cores)
                gpu_hashes = np.array([workload.msa_hash(msas[e]) for e in range(n_cpu)], np.uint64)
                same = bool(np.array_equal(gpu_hashes, hashes))
                extra["parity"] = {"ends_checked": int(n_cpu), "identical": same, "what": "per-end FNV-1a hash of the MSA bytes, GPU arm vs %s CPU arm" % kind}
                if not same:
                    bad = [int(i) for i in np.nonzero(gpu_hashes != hashes)[0][:8]]
                    sys.stderr.write("[bench] PARITY GATE FAILED: the GPU alignments of ends %s differ from the CPU reference's; no number is reported\n" % bad)
                    return 3
                c = float(np.sum(cells[:n_cpu]))
                best = min(secs.values())
                extra["cpu_baseline"] = {"value": c / best / 1e9, "unit": "Gcell/s", "ends_per_s": n_cpu / best, "cores": cores, "kind": kind,
                                         "sample": "first %d of the step's ends (8 x 2 kbp each), %.1f s wall, OpenMP schedule(dynamic,1) over ends" % (n_cpu, best),
                                         "allocator": {"glibc_default_gcells": c / secs["glibc_default"] / 1e9, "retained_blocks_gcells": c / secs["retained_blocks"] / 1e9,
                                                       "note": "retained_blocks = glibc told to keep and reuse large blocks, the stand-in for the jemalloc Cactus links"},
                                         "per_thread_gcells": c / best / 1e9 / cores}
            except Exception as e:  # noqa: BLE001
                extra["cpu_baseline"] = {"value": None, "unit": "Gcell/s", "cores": cores, "kind": "unavailable", "sample": str(e)}
        if not args.no_extras:
            try:
                extra["shapes"] = shapes_leg(eng)
            except Exception as e:  # noqa: BLE001
                extra["shapes"] = {"error": str(e)}
    stage.close()
    eng.close()
    if rank == 0 and not args.no_extras:
        # the end queue driven by 16 host threads, in a fresh process like the cPecan section below (this one has just run the reference
        # arm's allocator settings, OpenMP teams of two libraries and a dozen arena shapes; a clean process is what a Cactus run looks like)
        try:
            cmd = [sys.executable, os.path.abspath(__file__), "--flowers-only", str(max(8, n_ends // 4)), "--cells-per-end", repr(my_cells / max(1, n_ends))]
            env = dict(os.environ)
            env["LOCAL_RANK"] = str(local_rank)
            # 16 caller threads + the lanes' workers + the library's OpenMP team on a 16-CPU quota: idle OpenMP workers must sleep, not
            # spin (measured 131 vs 217 Gcell/s); the single-caller legs above keep the default policy (wake-ups cost them ~9 ms a step)
            env.setdefault("OMP_WAIT_POLICY", "passive")
            env["OMP_NUM_THREADS"] = str(usable_cores())
            for k in ("RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
                env.pop(k, None)
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
            fl = json.loads(out.stdout.strip().splitlines()[-1])
            fl["single_batch_e2e_gcells_per_s"] = my_cells / e2e_ms / 1e6 if e2e_ms == e2e_ms else None
            extra["e2e_flowers"] = fl
        except Exception as e:  # noqa: BLE001
            extra["e2e_flowers"] = {"error": str(e)}
    # ---- N > 1: the same host-buffer call IN ONE PROCESS over all N devices (one context, devices[] = 0..N-1; the ends are dealt by
    # estimated cost, results land in the caller's buffers, no gather); rank 0 drives, the other ranks idle at the barrier ----
    if world > 1 and not args.no_e2e and not args.no_extras:
        barrier()
        # (the other ranks must wait on the HOST: a rank parked in an NCCL barrier keeps a spinning kernel on its GPU, and a second process's
        # context on that GPU would be time-sliced against it)
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                eng_all = cb.Engine(cb.PoaParams(devices=list(range(world)), host_threads=cores))
                a_seq, a_lens, a_flat = workload.synth_ends(0, E * world, K_SEQS, L_BP)
                pins = [torch.from_numpy(a).pin_memory() for a in (a_seq, a_lens, a_flat)]
                q_nseq, q_lens, q_flat = [t.numpy() for t in pins]
                nA = E * world

                def all_once():
                    outs = (C.c_void_p * nA)()
                    ml = np.zeros(nA, np.int32)
                    cc = np.zeros(nA, np.int64)
                    eng_all._check(eng_all.lib.barb200_poa_msa_batch(eng_all.ctx, nA, q_nseq.ctypes.data, q_lens.ctypes.data, q_flat.ctypes.data, None, outs,
                                                                     ml.ctypes.data, cc.ctypes.data))
                    eng_all.lib.barb200_free_many(outs, nA)
                    return float(cc.sum())
                all_once()
                t2 = time.time()
                tot = 0.0
                for _ in range(args.steps):
                    tot = all_once()
                dt = (time.time() - t2) / args.steps
                extra["e2e_in_process"] = {"value": tot / dt / 1e9, "unit": "Gcell/s", "ms_per_step": dt * 1e3, "devices": world,
                                           "api": "ONE context over %d devices (barb200_params.devices[]), barb200_poa_msa_batch with host buffers, cost-sorted deal, no gather" % world}
                eng_all.close()
            except Exception as e:  # noqa: BLE001
                extra["e2e_in_process"] = {"error": str(e)}
            store.set("barb200_inproc_done", "1")
        else:
            store.wait(["barb200_inproc_done"])
        barrier()
    # ---- cPecan mode (its own context: the POA arenas are released first) ----
    pecan = None
    if args.pecan_pairs_per_step > 0:
        # measured in a fresh process per rank (its host-side phases ran several times slower inside this one after the POA
        # section; a clean process reproduces the stand-alone numbers), all ranks at the same time; reductions happen here
        cmd = [sys.executable, os.path.abspath(__file__), "--pecan-only", "--pecan-pairs-per-step", str(args.pecan_pairs_per_step),
               "--steps", str(args.steps), "--warmup", str(args.warmup), "--cpu-budget", str(args.cpu_budget)]
        cmd += ["--no-e2e"] if args.no_e2e else []
        cmd += ["--no-cpu-baseline"] if args.no_cpu_baseline else []
        cmd += ["--dump-outputs", args.dump_outputs] if args.dump_outputs and rank == 0 else []
        env = dict(os.environ)
        env["OMP_NUM_THREADS"] = str(host_threads)
        barrier()
        cp = subprocess.run(cmd, env=env, capture_output=True, text=True)
        mine = None
        for ln in cp.stdout.splitlines():
            if ln.startswith("PECAN_JSON "):
                mine = json.loads(ln[len("PECAN_JSON "):])
        failed = mine is None
        if failed:          # every rank still takes part in the reduction below; the section is reported as failed
            sys.stderr.write("[bench] the cPecan section failed on rank %d:\n%s\n" % (rank, cp.stderr[-2000:]))
            mine = {"dev_ms": float("inf"), "e2e_ms": float("inf"), "cells": 0.0, "n_pairs": 0, "launches": 0, "steps": 1, "h2d": 0, "d2h": 0, "same": False}
        mxp, smp = D.reduce_stats([mine["dev_ms"], mine["e2e_ms"], mine["cells"], float(mine["n_pairs"]), float(mine["launches"]), 1.0 if failed else 0.0], dev)
        if rank == 0:
            pecan = {"error": "the cPecan section failed on %d rank(s); see stderr" % int(smp[5])} if smp[5] > 0 else \
                pecan_object(mine, mxp, smp, args.pecan_pairs_per_step)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    dev_ms_max, wall_ms_max, e2e_ms_max = float(mx[0]), float(mx[1]), float(mx[2])
    tot_cells, tot_ends, tot_launches = float(sm[3]), float(sm[4]), int(sm[5])
    value = tot_cells * args.steps / dev_ms_max / 1e6          # Gcell/s
    peak, peak_src = measured_peak()
    # roofline of the dominant kernel: algorithmic bytes per launch / average launch duration, rank 0's launches
    step_ms = dev_ms / max(1, args.steps)
    achieved = my_cells * ALGO_BYTES_PER_CELL / (step_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    prof = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof))
            traffic = pj["dram_bytes_per_cell"] * my_cells
            traffic_src = "DERIVED, not measured in this run: %.2f DRAM bytes per cell (ncu --set full capture summarised in %s) x the cells of one step" % (
                pj["dram_bytes_per_cell"], pj["sources"][0])
        except Exception:  # noqa: BLE001
            traffic = None
    h2d = int(flat.nbytes + lens.nbytes * 2 + lens.size * 8 + n_seq.size * 40)
    calls = max(1, int(phases["calls"]))
    line = {"metric": METRIC, "value": value, "unit": "Gcell/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic", "config": config,
            "ends_per_s": tot_ends * args.steps / dev_ms_max * 1e3,
            "wall_ms_per_step": wall_ms_max / args.steps,
            "e2e": {"value": tot_cells / e2e_ms_max / 1e6, "unit": "Gcell/s", "ends_per_s": tot_ends / e2e_ms_max * 1e3,
                    "ms_per_step": e2e_ms_max, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h + n_ends * 16,
                    "api": "barb200_poa_msa_batch (host buffers: pack + guide trees + H2D + kernel + D2H + unpack)" +
                           (" + NCCL send/recv gather of the MSA bytes on rank 0" if world > 1 else ""),
                    "phases_rank0_ms": {k: phases[k] / calls for k in ("build_ms", "run_ms", "device_ms", "fetch_ms", "total_ms", "gather_ms")},
                    "host_threads_per_rank": host_threads},
            "gpu_launches": tot_launches, "buckets": buckets,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": "poa_msa_kernel_t128",
                         "bytes_per_cell_algorithmic": ALGO_BYTES_PER_CELL,
                         "frac_of_peak_really_moved": (traffic / (step_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "note": "algorithmic = SURVEY.md 8d's contract figure (five int32 planes written + three read per cell); the kernel itself stores "
                                 "8 B/cell, so frac > 1 means it beats what any implementation streaming those planes could do at peak. It is NOT HBM-bound: "
                                 "frac_of_peak_really_moved is the DRAM traffic it actually causes over the peak; the ncu capture (profiles/) shows issue slots "
                                 "47 % busy at 2.05 warp-instructions per cell, stalls split between the two barriers per row, L2 loads and dependent shuffles"},
            "clocks": sampler.summary(), "rank_checksums": checksums}
    line.update(extra)
    if pecan is not None:
        line["pecan"] = pecan
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ends-per-step", type=int, default=int(os.environ.get("BARB200_ENDS_PER_STEP", "2368")),
                    help="ends per GPU per step (default 16 x 148 SMs)")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (and with it the parity gate)")
    ap.add_argument("--no-extras", action="store_true", help="skip the shapes / e2e_flowers / in-process multi-GPU legs")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer legs (for runs under ncu: the streamed e2e path releases jobs "
                    "to a RUNNING kernel from the host, which deadlocks under ncu's kernel serialisation)")
    ap.add_argument("--workload", default=None, help="replay a record made by shim/cactus_bar_harvest.c (BARB200_HARVEST=<file> during a reference "
                    "bar() run) instead of the synthetic workload")
    ap.add_argument("--flowers-only", type=int, default=0, help="internal: this process only runs the e2e_flowers leg over that many flowers and prints its numbers")
    ap.add_argument("--cells-per-end", type=float, default=0.0, help="internal (with --flowers-only)")
    ap.add_argument("--pecan-only", action="store_true", help="internal: this process only measures the cPecan section and prints its raw numbers")
    ap.add_argument("--pecan-pairs-per-step", type=int, default=int(os.environ.get("BARB200_PECAN_PAIRS_PER_STEP", "4736")),
                    help="cPecan-mode pairs per GPU per step (default 32 x 148 SMs); 0 skips the cPecan section")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed POA and cPecan steps returned in their last step as DIR/<name>.npy (float32 / float64; "
                         "per-end and per-pair summaries of the whole step, full alignments of a fixed sample); GPU arm, rank 0")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    if args.flowers_only:
        import cactus_b200 as cb
        eng = cb.Engine(cb.PoaParams(device=int(os.environ.get("LOCAL_RANK", "0")), host_threads=usable_cores()))
        fl, _ = flowers_leg(eng, 5000000, args.flowers_only, 16, args.cells_per_end)
        eng.close()
        print(json.dumps(fl))
        return 0
    if args.pecan_only:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        host_threads = int(os.environ.get("OMP_NUM_THREADS", "0")) or max(1, usable_cores() // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))))
        m = pecan_measure(local_rank, rank, rank * args.pecan_pairs_per_step, args.pecan_pairs_per_step, args.steps, args.warmup,
                          min(args.cpu_budget, 12.0), not args.no_cpu_baseline, args.no_e2e, host_threads, args.dump_outputs)
        print("PECAN_JSON " + json.dumps(m))
        return 0
    if args.impl == "reference":
        return reference_arm(args) if rank == 0 else 0     # the reference's CPU implementation; rank 0 only
    if args.workload:
        return replay_arm(args) if rank == 0 else 0
    return gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
