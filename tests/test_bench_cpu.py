"""bench.py's host-side logic (no GPU): workload split and FLOP accounting, and the reference arm - the UNMODIFIED reference's
engine on the host cores - printing the contract's JSON line."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_split_and_schedules():
    assert bench.split_counts(100, 8) == [13, 13, 13, 13, 12, 12, 12, 12] and bench.split_counts(100, 4) == [25] * 4
    assert sum(bench.split_counts(100, 3)) == 100 and bench.split_counts(20, 1) == [20]
    upd, ren = bench.chain_schedule(20)
    assert upd[0] == (2, 1) and upd[1:] == [(1, m) for m in range(2, 20)] and ren == [(20, 20)]
    # sharded rounds: every view is stored exactly once, a round's views see the memory of the previous rounds only
    for counts in ([13, 13, 13, 13, 12, 12, 12, 12], [50, 50], [3, 2, 1]):
        upd, ren = bench.sharded_schedule(counts)
        assert sum(n for n, _ in upd) == sum(counts) and ren == [(sum(counts), sum(counts))]
        seen = 2
        i = 1
        for s in range(max(counts)):
            part = sum(1 for r, c in enumerate(counts) if s < c and not (r == 0 and s < 2))
            assert all(m == seen for _, m in upd[i:i + part])
            i += part
            seen += part
    # SURVEY.md 8a per-view figures: C3 = 20 x 523.0 GF encoder + updates + render of 20 views against 20
    f = bench.job_flops(512, 20, *bench.chain_schedule(20))
    want = 20 * 523.0e9 + 2 * (177.3e9 + 50.7e9 + 21.74e9) + sum(177.3e9 + 50.7e9 + 21.74e9 * m for m in range(2, 20)) + 20 * (177.3e9 + 21.74e9 * 20)
    assert abs(f - want) / want < 1e-12 and 31.0e12 < f < 32.0e12


def test_dump_outputs_whole_or_fixed_sample(tmp_path):
    """--dump-outputs: the per-view result dicts stacked over views, float32; within the budget the arrays are written
    whole, above it every file holds the same sample of its array on every run and the files stay within the budget."""
    import numpy as np
    import torch
    g = torch.Generator().manual_seed(0)
    out = [{"pts3d": torch.randn(4, 5, 3, generator=g), "conf": torch.rand(4, 5, generator=g, dtype=torch.float64)} for _ in range(3)]
    full = {k: torch.stack([d[k] for d in out]).float().numpy() for k in ("pts3d", "conf")}
    assert bench.dump_outputs(out, str(tmp_path / "whole")) == ["conf", "pts3d"]
    for k, want in full.items():
        got = np.load(tmp_path / "whole" / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, want)
    for run in ("a", "b"):
        bench.dump_outputs(out, str(tmp_path / run), budget=200)
    a = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in full}
    assert sum(v.nbytes for v in a.values()) <= 200 and all(v.size > 0 and v.dtype == np.float32 for v in a.values())
    for k, v in a.items():
        assert np.array_equal(v, np.load(tmp_path / "b" / f"{k}.npy")) and np.isin(v, full[k]).all()


@pytest.mark.timeout(600)
def test_reference_arm_prints_the_contract_line():
    from baseline import ref_loader
    if not ref_loader.available():
        pytest.skip("the reference is not installed under oracle/_ref")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c2", "--steps", "1",
                          "--warmup", "1", "--cpu-views", "2"], capture_output=True, text=True, timeout=500)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "views/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["same_config"] is False and line["config"]["cap"]
