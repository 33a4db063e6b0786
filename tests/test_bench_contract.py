"""bench.py's output contract on the leg that runs without a GPU: `--impl reference` prints ONE JSON line with the keys the
driver reads (metric / value / unit / impl / cpu_baseline / e2e ...), for the POA section and the cPecan section."""
import json
import os
import subprocess
import sys

import pytest

import _reflib as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not (R.have_ref() and R.have_pecan_ref()), reason="oracle/_ref not built (needs the reference's sources, see oracle/Makefile)")
def test_reference_arm_prints_one_json_line():
    cp = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                         "--cpu-budget", "1", "--ends-per-step", "8", "--pecan-pairs-per-step", "8"],
                        capture_output=True, text=True, timeout=600)
    assert cp.returncode == 0, cp.stderr[-2000:]
    lines = [ln for ln in cp.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, cp.stdout[-2000:]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Gcell/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"]
    assert d.get("product_library_loaded") is False            # the reference arm maps no product code
    assert d["cpu_baseline"]["allocator"]["glibc_default_gcells"] > 0 and d["cpu_baseline"]["allocator"]["retained_blocks_gcells"] > 0
    p = d["pecan"]
    assert p["impl"] == "reference" and p["value"] > 0 and p["cpu_baseline"]["kind"] == "reference"
