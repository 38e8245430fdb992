"""Checks of the benchmark's interface: build() is callable, the reference arm of bench.py prints exactly one JSON line
with the keys a reader of the result expects, and (on a GPU) --dump-outputs writes the results of the timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_build_entry_point():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.build()  # make is a no-op when the library is current; raises if the library cannot be produced or loaded
    assert callable(g.smoke)


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-procs", "4"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "candidates/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1 and d["dtype"] == "f64"
    staged = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "gpExp"))  # the unmodified reference, when build() staged it
    assert d["cpu_baseline"]["kind"] == ("reference" if staged else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["scaling"] == "strong" and d["config"]["candidates_total"] == 100000
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_cpu_legs_of_the_other_configs_print_one_json_line():
    """`--impl reference-configs` (called by the GPU arm at N = 1): bounded samples of cfg-1 / cfg-3 / cfg-4 through the
    staged unmodified reference, or one line saying it is not staged."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference-configs"], capture_output=True,
                         text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "gpExp")):
        assert "unavailable" in d
        return
    assert d["kind"] == "reference" and d["cores"] >= 1
    for cfg in ("cfg1", "cfg3", "cfg4"):
        assert d[cfg]["candidates_per_s_per_step"] > 0 and d[cfg]["seconds"] < 120 and d[cfg]["sample"]


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_step(tmp_path):
    """--dump-outputs: the 256 picks of the timed step, their costs and pivots, and the cost of every candidate, as float64;
    the last pick is the arg-min of those costs.  --quick-design keeps the run short (same state shape, random design)."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--quick-design", "--no-cpu",
                          "--no-configs", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 1
    z = {n: np.load(tmp_path / f"{n}.npy") for n in ("indices", "pick_scores", "pivots", "scores")}
    assert all(a.dtype == np.float64 for a in z.values())
    assert z["indices"].shape == z["pick_scores"].shape == z["pivots"].shape == (256,) and z["scores"].shape == (100_000,)
    last = int(z["indices"][-1])
    assert z["scores"][last] == z["scores"].min() == z["pick_scores"][-1]
    assert np.all(np.isfinite(z["scores"])) and z["pivots"][-1] > 0
