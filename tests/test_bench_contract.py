"""bench.py contract: the reference arm runs without a GPU and prints one JSON line with the agreed keys; --dump-outputs
writes the GPU arm's results of its last timed step, the same on every run with the same arguments."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1", "--sims", "6", "--ref-segment", "3"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "sims/s" and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
    assert "workload" in line["config"]
    # a step is a segment of consecutive simulations of one search; the sample says so, and the arm reports how many
    # simulations ended on a terminal node (the same statistic the GPU arm prints)
    assert "3 consecutive simulations of a 6-simulation search" in line["config"]["sample"]
    assert 0.0 <= line["config"]["terminal_leaf_fraction"] < 1.0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_samples_a_large_result_within_the_budget(tmp_path):
    """A result above the size limit is cut to the same seeded sample of games on every call, rows kept whole."""
    import numpy as np

    import bench
    G = 40000
    arrays = {"visit_counts": np.arange(G * 256, dtype=np.uint32).reshape(G, 256), "n_children": np.arange(G, dtype=np.uint32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES
    got = {f.name: np.load(f) for f in (tmp_path / "a").iterdir()}
    assert {f.name for f in (tmp_path / "b").iterdir()} == set(got)
    assert all(np.array_equal(np.load(tmp_path / "b" / n), a) for n, a in got.items())
    keep = got["game_index.npy"].astype(np.int64)
    assert 0 < len(keep) < G and np.all(np.diff(keep) > 0)
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["visit_counts.npy"], arrays["visit_counts"][keep])
    assert np.array_equal(got["n_children.npy"], keep)


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
@pytest.mark.parametrize("game,sims", [("c4", 64), ("chess", 16)])
def test_dump_outputs_are_the_last_steps_root_children_and_reproducible(tmp_path, game, sims):
    """Two runs with the same arguments write identical arrays: the root children of every game after `sims` simulations."""
    import numpy as np
    G = 128
    dumps = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--game", game, "--games", str(G), "--sims", str(sims),
                            "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--full-game-moves", "0", "--dump-outputs", str(tmp_path / d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        dumps.append({f.name: np.load(f) for f in (tmp_path / d).iterdir()})
    a, b = dumps
    moves = "actions.npy" if game == "c4" else "moves.npy"
    assert set(a) == {moves, "visit_counts.npy", "child_ids.npy", "n_children.npy", "game_index.npy"}
    assert all(np.array_equal(a[n], b[n]) for n in a)
    assert np.array_equal(a["game_index.npy"], np.arange(G))
    assert np.all(a["visit_counts.npy"].sum(axis=1) == sims - 1)          # every root is ongoing: one simulation expands it
    assert np.all(a["n_children.npy"] >= 1)
