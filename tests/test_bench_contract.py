"""bench.py's output contract on CPU: the reference arm (the only arm that runs without a GPU) prints exactly ONE JSON
line on stdout with the keys the driver reads, and the product arm refuses to run without a CUDA device instead of
falling back to the CPU."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
  e = dict(os.environ)
  e.pop("WORLD_SIZE", None); e.pop("RANK", None)
  e.update(env or {})
  return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e,
                        timeout=600)


def test_reference_arm_prints_one_json_line():
  r = _run("--impl", "reference", "--steps", "3", "--warmup", "1")
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.strip()]
  assert len(lines) == 1, r.stdout
  d = json.loads(lines[0])
  assert d["impl"] == "reference" and d["unit"] == "maps/s" and d["higher_is_better"] is True
  assert d["value"] > 0 and d["steps"] == 3 and d["dtype"] == "f32" and d["data"] == "synthetic"
  # the unmodified reference is the line whenever it is importable (/root/reference here, baseline/_ref on the GPU
  # box), with the C / OpenMP port next to it; otherwise the port is the line
  assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
  if d["cpu_baseline"]["kind"] == "reference":
    assert d["port"]["kind"] == "port" and d["port"]["value"] > 0
  else:
    assert "reference_note" in d
  assert "units_per_step" not in d["config"]       # same config keys as the product arm's line
  assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
  assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
  assert "config 2" in d["config"]["workload"] and d["vs_baseline"] is None


def test_reference_arm_other_ranks_stay_silent():
  r = _run("--impl", "reference", "--gpus", "2", "--steps", "3", env={"RANK": "1", "WORLD_SIZE": "2"})
  assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a box without a GPU")
def test_product_arm_has_no_cpu_path():
  r = _run("--steps", "3")
  assert r.returncode != 0 and "needs a CUDA device" in (r.stderr + r.stdout)


def test_dump_outputs_fits_the_budget_at_fixed_positions(tmp_path, monkeypatch):
  import bench
  monkeypatch.setattr(bench, "DUMP_BYTES", 7 * 4000)
  top = torch.arange(2 * 3 * 40 * 50, dtype=torch.float32).view(2, 3, 40, 50)
  top[top % 5 == 0] = -math.inf    # the fill of unobserved cells
  top[top % 7 == 0] = math.nan
  top[top % 11 == 0] = math.inf
  hgt = top[:, :1].expand(2, 3, 40, 50)
  arrays = {"topdown": top, "mask": top % 3 == 0, "height": hgt, "offset": torch.tensor([1.5], dtype=torch.float64)}
  bench.dump_outputs(arrays, str(tmp_path / "a"))
  bench.dump_outputs(arrays, str(tmp_path / "b"))
  files = sorted(f.name for f in (tmp_path / "a").iterdir())
  assert files == sorted(["topdown.npy", "topdown_nonfinite.npy", "mask.npy", "height.npy", "height_nonfinite.npy",
                          "offset.npy", "offset_nonfinite.npy"])
  assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 7 * 4000 + 7 * 128
  for f in files:
    got = np.load(tmp_path / "a" / f)
    assert got.dtype in (np.float32, np.float64) and np.isfinite(got).all(), f
    assert np.array_equal(got, np.load(tmp_path / "b" / f)), f
  pos = bench.dump_positions(top.numel(), 4000 // 4)
  for name, want in (("topdown", top), ("height", hgt)):
    want = want.reshape(-1).numpy()[pos]
    got, flag = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "a" / f"{name}_nonfinite.npy")
    decoded = np.where(flag == 1, np.inf, np.where(flag == -1, -np.inf, np.where(flag == 2, np.nan, got)))
    assert np.array_equal(decoded, want, equal_nan=True) and (flag != 0).any() and (flag == 0).any()
  assert np.array_equal(np.load(tmp_path / "a" / "mask.npy"), (top % 3 == 0).float().reshape(-1).numpy()[pos])
  offset = np.load(tmp_path / "a" / "offset.npy")
  assert offset.dtype == np.float64 and offset.tolist() == [1.5]


def test_bad_arguments_are_refused():
  assert _run("--steps", "0").returncode != 0
  assert _run("--impl", "reference", "--dump-outputs", "x").returncode != 0


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["proj", "flow", "builder"])
def test_dumped_outputs_repeat_from_run_to_run(workload, tmp_path):
  """Same arguments, same inputs: two runs dump the same arrays, within the size limit, after exactly --steps steps."""
  args = ("--workload", workload, "--steps", "2", "--warmup", "1", "--no-extra", "--no-cpu-baseline", "--e2e-steps", "0")
  for run in ("a", "b"):
    r = _run(*args, "--dump-outputs", str(tmp_path / run))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
  files = sorted(p.name for p in (tmp_path / "a").iterdir())
  assert files and files == sorted(p.name for p in (tmp_path / "b").iterdir())
  assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64 << 20
  for f in files:
    a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
    assert a.dtype in (np.float32, np.float64) and a.size > 0 and np.isfinite(a).all(), f
    assert a.tobytes() == b.tobytes(), f
