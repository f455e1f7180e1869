"""bench.py contract pieces that can run without a GPU: the reference (CPU) arm's JSON line, the synthetic generator's
determinism and the roofline arithmetic."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")      # what torchrun sets for its children
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                          "--steps", "2", "--warmup", "1", "--gpus", "1"], capture_output=True, text=True, env=env, check=True).stdout
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "events/s" and d["higher_is_better"] is True
    assert d["metric"] == "CCO train events/sec to indicator model"
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and "sample" in cb
    assert cb["cores"] == len(os.sched_getaffinity(0))           # all host threads, not OMP_NUM_THREADS=1


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", "--gpus", "2"],
                       capture_output=True, text=True, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_synthetic_generator_is_deterministic_and_binary():
    import synth
    a, b = synth.make("tiny"), synth.make("tiny")
    for (nr, nc, rp, ci), (_, _, rp2, ci2) in zip(a.mats, b.mats):
        assert np.array_equal(rp, rp2) and np.array_equal(ci, ci2)
        assert rp[0] == 0 and (np.diff(rp) >= 0).all() and len(ci) == rp[-1]
        for r in range(0, nr, 37):
            row = ci[rp[r]:rp[r + 1]]
            assert (np.diff(row) > 0).all()                        # sorted, no duplicates
    assert a.mats[0][3].tolist() != a.mats[1][3].tolist()          # event types differ (seed 1234 + t)


def test_min_events_per_user_shrinks_the_user_space_like_preparator():
    import synth
    w = synth.make("tiny", min_events_per_user=25)
    raw = synth.make("tiny")
    assert w.n_users < raw.n_users
    assert all(m[0] == w.n_users for m in w.mats)                  # one shared, compacted row space


def test_algorithmic_bytes_formula():
    sys.path.insert(0, ROOT)
    import bench

    class St:
        nnz_downsampled = [1000, 2000]
        products = [50_000, 70_000]
        distinct_cells = [40_000, 60_000]
        out_nnz = [3_000, 4_000]
    # SURVEY.md 8(d): 4 nnz(A') + 8 (I_A+1) + 8 nnz(A') + 4 P + 4 C + 4 I_A + 12 out
    assert bench.algorithmic_bytes(St, 1, 100) == 4 * 1000 + 8 * 101 + 8 * 1000 + 4 * 70_000 + 4 * 60_000 + 4 * 100 + 12 * 4_000


def _read_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_samples_whole_rows_under_the_size_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    rng = np.random.default_rng(1)
    n_rows, k = 20_000, 50
    model = []
    for _ in range(3):
        rp = np.concatenate([[0], np.cumsum(rng.integers(0, k + 1, n_rows))]).astype(np.int64)
        model.append((0, n_rows, n_rows, rp, rng.integers(0, n_rows, rp[-1]).astype(np.int32), rng.random(rp[-1]),
                      np.zeros(0, np.int32)))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), model, model, k)
    a, b = _read_dump(tmp_path / "a"), _read_dump(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[n], b[n]) for n in a)          # a fixed sample
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= (1 << 20) + 4096
    assert all(x.dtype == np.float64 for x in a.values())
    rows = a["rows"].astype(np.int64)
    assert 0 < len(rows) < n_rows and (np.diff(rows) > 0).all()
    for i, (_, _, _, rp, ci, ll, _) in enumerate(model):
        want = np.concatenate([np.arange(rp[r], rp[r + 1]) for r in rows])
        assert np.array_equal(a[f"indicator{i}_row_len"], np.diff(rp)[rows])
        assert np.array_equal(a[f"indicator{i}_resident_row_len"], np.diff(rp)[rows])
        assert np.array_equal(a[f"indicator{i}_col_idx"], ci[want]) and np.array_equal(a[f"indicator{i}_llr"], ll[want])


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_and_match_the_oracle(orc, tmp_path):
    import synth
    for d in ("a", "b"):
        subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "2", "--warmup", "1",
                        "--cpu-sample", "none", "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, check=True)
    a, b = _read_dump(tmp_path / "a"), _read_dump(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[n], b[n]) for n in a)
    w = synth.make("tiny")
    ref = orc.train([orc.Csr(*m) for m in w.mats], [orc.Params(*p) for p in w.params], 42)
    assert np.array_equal(a["rows"], np.arange(w.n_items))                                # tiny: every row is written
    for i, r in enumerate(ref):
        assert np.array_equal(a[f"indicator{i}_row_len"], np.diff(r.row_ptr))
        assert np.array_equal(a[f"indicator{i}_resident_row_len"], np.diff(r.row_ptr))
        assert np.array_equal(a[f"indicator{i}_col_idx"], r.col_idx)
        assert np.allclose(a[f"indicator{i}_llr"], r.llr, rtol=1e-6, atol=0)
