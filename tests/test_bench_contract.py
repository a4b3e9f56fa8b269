"""bench.py's reference arm (the CPU port of the path on the host cores, the one other place besides tests / smoke that may
execute oracle/) prints the contract's JSON line without touching a GPU; the B200 arm refuses to run without one, and
its --dump-outputs writes the timed move's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUTPUT_NAMES = ("actions", "root_value", "child_visits", "init_value")


def _run(*flags):
  return subprocess.run([sys.executable, os.path.join(REPO, "bench.py")] + list(flags), capture_output=True, text=True,
                        timeout=600, cwd=REPO)


def test_reference_arm_prints_the_contract_line():
  r = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--games", "64", "--sims", "5", "--ref-moves-per-step", "1")
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.strip()]
  assert len(lines) == 1  # ONE JSON line on stdout
  d = json.loads(lines[0])
  assert d["impl"] == "reference" and d["metric"] == "mcts_node_expansions_per_sec" and d["unit"] == "expansions/s"
  assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
  assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
  assert d["config"]["workload"].startswith("C4") and d["config"]["games_per_gpu"] == 64
  assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
  assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_b200_arm_needs_a_gpu():
  import torch
  if torch.cuda.is_available():
    return
  r = _run("--steps", "1", "--warmup", "0", "--no-cpu-baseline")
  assert r.returncode != 0 and "GPU" in (r.stderr + r.stdout)  # no CPU fallback for the product path


def test_dump_outputs_samples_the_same_games_past_the_size_cap(tmp_path, monkeypatch):
  import bench
  G, A = 1000, 18
  rng = np.random.default_rng(3)
  outputs = {"actions": rng.integers(0, A, G).astype(np.float64), "root_value": rng.normal(size=G),
             "child_visits": rng.random((G, A)), "init_value": rng.normal(size=G).astype(np.float32)}
  bench.dump_outputs(str(tmp_path / "whole"), outputs)
  for name, a in outputs.items():
    got = np.load(tmp_path / "whole" / (name + ".npy"))
    assert got.dtype == a.dtype and np.array_equal(got, a)
  assert not (tmp_path / "whole" / "game_index.npy").exists()
  monkeypatch.setattr(bench, "DUMP_BYTES", 20_000)
  for run in ("a", "b"):
    bench.dump_outputs(str(tmp_path / run), outputs)
  keep = np.load(tmp_path / "a" / "game_index.npy").astype(np.int64)
  assert 0 < len(keep) < G and np.all(np.diff(keep) > 0)
  assert sum(np.load(tmp_path / "a" / (n + ".npy")).nbytes for n in OUTPUT_NAMES + ("game_index",)) <= 20_000
  for name, a in outputs.items():  # the same games in every array, and the same sample in every run
    assert np.array_equal(np.load(tmp_path / "a" / (name + ".npy")), a[keep])
    assert np.array_equal(np.load(tmp_path / "b" / (name + ".npy")), a[keep])


def test_dump_outputs_needs_the_b200_arm(tmp_path):
  r = _run("--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path))
  assert r.returncode != 0 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_same_move_whatever_the_step_count(tmp_path):
  """Every timed step plays the same move from the same resident inputs, so runs that time it 1 and 3 times write
  identical outputs, and those are a valid move: actions among the legal ones, visit distributions summing to 1."""
  G, A = 512, 18
  quick = ["--games", str(G), "--sims", "10", "--actions", str(A), "--warmup", "1", "--no-cpu-baseline", "--no-sweep",
           "--no-conv", "--no-f32", "--no-selfplay", "--no-concurrent"]
  dumps = []
  for steps in (1, 3):
    d = tmp_path / ("steps%d" % steps)
    r = _run(*quick, "--steps", str(steps), "--dump-outputs", str(d))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == steps
    assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in OUTPUT_NAMES)
    dumps.append({n: np.load(d / (n + ".npy")) for n in OUTPUT_NAMES})
  one, three = dumps
  for n in OUTPUT_NAMES:
    assert np.array_equal(one[n], three[n]), n
  assert one["actions"].shape == (G,) and one["actions"].dtype == np.float64
  assert np.all((one["actions"] >= 0) & (one["actions"] < A) & (one["actions"] == np.round(one["actions"])))
  assert one["child_visits"].shape == (G, A) and one["child_visits"].dtype == np.float64
  assert np.allclose(one["child_visits"].sum(1), 1.0)
  assert one["root_value"].dtype == np.float64 and one["init_value"].dtype == np.float32
  assert np.all(np.isfinite(one["root_value"])) and np.all(np.isfinite(one["init_value"]))
