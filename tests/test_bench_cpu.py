"""Host-side pieces of bench.py that need no GPU: the reference arm's line (bench.py --impl reference, the restated C
control flow on the host cores) and the watchdog over the legs that follow the timed region."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_tail_guard_prints_the_line_when_a_leg_stalls():
    code = (
        "import sys, time; sys.path.insert(0, %r); import bench\n"
        "out = {'metric': 'm', 'value': 1.0, 'e2e': None}\n"
        "g = bench.TailGuard(0, out, 0.3); g.leg = 'e2e'\n"
        "time.sleep(30)\n"
        "print('not reached')\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["value"] == 1.0 and "e2e" in line["tail_note"]


def test_tail_guard_is_silent_when_the_legs_finish():
    code = (
        "import sys, time; sys.path.insert(0, %r); import bench\n"
        "out = {'metric': 'm', 'value': 2.0}\n"
        "g = bench.TailGuard(0, out, 30.0); out['e2e'] = {'value': 3.0}; g.finish()\n"
        "w = bench.TailGuard(1, None, 30.0); w.finish()\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0]) == {"metric": "m", "value": 2.0, "e2e": {"value": 3.0}}


def test_dump_outputs_writes_every_result_as_float64(tmp_path, monkeypatch):
    """--dump-outputs: a, var(a), the pick and the rows of K (all of them when K fits the budget, else a seeded sample)."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    n, L = 40, 1000
    g = torch.Generator().manual_seed(0)
    K = torch.randn(n, n, dtype=torch.float64, generator=g)
    a, vara = torch.randn(L, dtype=torch.float64, generator=g), torch.rand(L, dtype=torch.float64, generator=g)
    res = (torch.tensor([3.5], dtype=torch.float64), torch.tensor([17]))
    bench.dump_outputs(str(tmp_path / "all"), torch, K, a, vara, res)
    monkeypatch.setattr(bench, "DUMP_K_BYTES", 8 * n * 5)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), torch, K, a, vara, res)
    load = lambda d, name: np.load(tmp_path / d / (name + ".npy"))
    for d in ("all", "s1"):
        got = {f.name for f in (tmp_path / d).iterdir()}
        assert got == {x + ".npy" for x in ("a", "vara", "K_rows", "K_rows_index", "picked_marker", "picked_tsq")}
        assert all(load(d, f[:-4]).dtype == np.float64 for f in got)
        assert np.array_equal(load(d, "a"), a.numpy()) and np.array_equal(load(d, "vara"), vara.numpy())
        assert load(d, "picked_marker").tolist() == [17.0] and load(d, "picked_tsq").tolist() == [3.5]
        rows = load(d, "K_rows_index").astype(np.int64)
        assert np.array_equal(load(d, "K_rows"), K.numpy()[rows])
    assert np.array_equal(load("all", "K_rows_index"), np.arange(n))
    sample = load("s1", "K_rows_index")
    assert len(sample) == 5 and np.all(np.diff(sample) > 0) and np.array_equal(sample, load("s2", "K_rows_index"))


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()


def test_reference_arm_line_on_the_small_workload():
    """--impl reference at the n = 2,000 shape: one JSON line, the keys the driver reads."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
