"""The oracle's sum / mean / prod scatter (oracle/dm_oracle.c: dmo_scatter) against the reference's own semantics,
and tests/_ordered.orth_project_ordered against the reference's orth_project outputs.  CPU only.

The reference reduces through torch_scatter with an `out=` canvas; oracle/ref_shim.py restates those calls as plain
torch functions (scatter_reduce_ for sum / prod, torch_scatter's scatter_mean source for mean).  Here they run on
torch CPU on random cases far larger and stranger than the fixtures: every GPU test of these reductions compares
with the oracle, so the oracle must first agree with the reference bit for bit.
"""
import numpy as np
import pytest
import torch

from oracle import dm_oracle as orc
from oracle import ref_shim
from tests import _ordered
from tests._golden import Golden, assert_same

PITCH = _ordered.PITCH


def shim_scatter(values, coords, valid, canvas, fill_value, reduction):
  """utils.py:389-492 (2-D canvas) on torch CPU through the shim's scatter functions: points that are masked or
  out of range go to a spare cell past the end of the row, which is dropped afterwards."""
  values = np.asarray(values, np.float32)
  Mh, Mw = canvas.shape[-2:]
  M = Mh * Mw
  lead = values.shape[:-1]
  rows = int(np.prod(lead))
  N = values.shape[-1]
  co = np.broadcast_to(coords, lead + (N, 2)).reshape(rows, N, 2)
  r, c = co[..., 0], co[..., 1]
  ok = (r >= 0) & (r < Mh) & (c >= 0) & (c < Mw)
  if valid is not None:
    ok &= np.broadcast_to(valid, values.shape).reshape(rows, N).astype(bool)
  index = torch.from_numpy(np.ascontiguousarray(np.where(ok, r * Mw + c, M)))
  src = torch.from_numpy(np.ascontiguousarray(values.reshape(rows, N)))
  before = torch.from_numpy(np.broadcast_to(canvas, lead + (Mh, Mw)).astype(np.float32).reshape(rows, M))
  if fill_value is not None:
    before = torch.full_like(before, float(fill_value))
  out = torch.cat((before, torch.zeros(rows, 1)), 1)
  if reduction == "mean":
    ref_shim._mean(src, index, dim=-1, out=out)
  else:
    ref_shim._make(reduction)(src, index, dim=-1, out=out)
  out = out[:, :M]
  mask = torch.nan_to_num((out - before).abs()) != 0  # utils.py:489-491
  return out.numpy().reshape(lead + (Mh, Mw)), mask.numpy().reshape(lead + (Mh, Mw))


def check_against_shim(values, coords, valid, canvas, fill, red, what):
  want = shim_scatter(values, coords, valid, canvas, fill, red)
  got = orc.scatter(values, coords, valid, canvas, fill, red)
  assert_same(got[0], want[0], f"{what} values")
  assert_same(got[1], want[1], f"{what} mask")
  return got


@pytest.mark.parametrize("seed", range(16))
def test_scatter_random_matches_shim(seed):
  values, coords, valid, canvas, fill, red = _ordered.scatter_case(4100 + seed)
  got = check_against_shim(values, coords, valid, canvas, fill, red, f"seed {seed} {red} fill={fill}")
  if red == "sum" and fill is None:
    assert _ordered.sum_bound_violations(got[0], values, coords, valid, canvas) == 0


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
def test_scatter_million_points_matches_shim(red):
  """10^6 points: 3 rows into a 2x3 canvas (about 1.7 * 10^5 hits a cell) and into a 300x300 one."""
  rng = np.random.default_rng(17)
  N = 1_000_000 // 3
  lo, hi = (0.999, 1.001) if red == "prod" else (-3.0, 3.0)
  values = rng.uniform(lo, hi, size=(3, N)).astype(np.float32)
  for Mh, Mw in ((2, 3), (300, 300)):
    coords = np.stack((rng.integers(-1, Mh + 1, (3, N)), rng.integers(-1, Mw + 1, (3, N))), -1)
    canvas = rng.uniform(-1, 1, (3, Mh, Mw)).astype(np.float32)
    for fill in (None, 1.0 if red == "prod" else 0.0):
      got = check_against_shim(values, coords, None, canvas, fill, red, f"{red} {Mh}x{Mw} fill={fill}")
      if red == "sum":
        assert _ordered.sum_bound_violations(got[0], values, coords, None,
                                             canvas if fill is None else np.full_like(canvas, fill)) == 0


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
def test_scatter_special_values_match_shim(red):
  """NaN, +-inf and -0.0 among the values; fills 0 / 1 / -inf / NaN and the caller's canvas (with specials too)."""
  rng = np.random.default_rng(23)
  Mh, Mw, N = 4, 5, 600
  values = _ordered.special_values((2, 3, N), 24, 0.5, 1.5, rate=0.05)
  coords = np.stack((rng.integers(0, Mh, (2, 1, N)), rng.integers(0, Mw, (2, 1, N))), -1)
  valid = rng.random((2, 1, N)) > 0.1
  canvas = _ordered.special_values((2, 3, Mh, Mw), 25, -1.0, 1.0, rate=0.2)
  for fill in (None, 0.0, 1.0, -np.inf, np.nan, -0.0):
    check_against_shim(values, coords, valid, canvas, fill, red, f"{red} fill={fill}")


def test_scatter_cancelling_sums_keep_mask_false():
  """+-x pairs whose sum returns exactly to the fill (or to the caller's value): the cell was hit but did not change,
  so its mask bit is False — for the sum and for the mean (0 / n = 0)."""
  Mh, Mw = 3, 4
  x = np.asarray([1.5, 0.25, 1e30, 3.0], np.float32)
  values = np.concatenate((x, -x, x[:2], -x[:2]))[None]           # (1, 12)
  cells = np.asarray([0, 5, 7, 11] * 2 + [2, 2, 2, 2])
  coords = np.stack((cells // Mw, cells % Mw), -1)[None]
  canvas = np.zeros((1, Mh, Mw), np.float32)
  canvas[0, 1, 1] = 7.0
  for red, fill in (("sum", 0.0), ("sum", None), ("mean", 0.0)):
    cv, m = check_against_shim(values, coords, None, canvas, fill, red, f"{red} fill={fill}")
    assert not m.any(), f"{red} fill={fill}: a cell whose sum returned to its start is marked changed"
    assert (cv == (canvas if fill is None else fill)).all()
  cv, m = check_against_shim(values, coords, None, canvas, None, "mean", "mean fill=None")  # 7 / 2 hits: changed
  assert m[0, 1, 1] and m.sum() == 1 and cv[0, 1, 1] == 3.5
  # the other direction: a sum that leaves the fill and a sum that lands on it from elsewhere
  values = np.asarray([[2.0, -2.0, 0.5]], np.float32)
  coords = np.asarray([[[0, 0], [0, 0], [1, 1]]])
  cv, m = check_against_shim(values, coords, None, canvas, -0.5, "sum", "sum onto fill")
  assert m[0, 1, 1] and cv[0, 1, 1] == 0.0 and not m[0, 0, 0]


def test_scatter_prod_through_zero_and_inf():
  values = np.asarray([[2.0, 0.0, 3.0, np.inf, -1.0, np.inf, 0.5, -0.0, -np.inf, 4.0]], np.float32)
  cells = np.asarray([0, 0, 1, 1, 1, 2, 2, 3, 3, 4])
  coords = np.stack((np.zeros_like(cells), cells), -1)[None]
  canvas = np.asarray([[[1.0, 5.0, -2.0, 0.0, np.inf, 1.0]]], np.float32)
  for fill in (1.0, None, 0.0, -np.inf):
    cv, _ = check_against_shim(values, coords, None, canvas, fill, "prod", f"prod fill={fill}")
  cv, m = orc.scatter(values, coords, None, canvas, 1.0, "prod")
  assert cv[0, 0, 0] == 0.0 and cv[0, 0, 1] == -np.inf and np.isnan(cv[0, 0, 3])


@pytest.mark.parametrize("Mh,Mw", [(1, 1), (1, 2), (2, 1), (3, 7), (17, 1), (300, 300)])
def test_scatter_canvas_sizes_match_shim(Mh, Mw):
  rng = np.random.default_rng(Mh * 1000 + Mw)
  N = 4000
  coords = np.stack((rng.integers(-1, Mh + 1, (2, N)), rng.integers(-1, Mw + 1, (2, N))), -1)
  valid = rng.random((2, N)) > 0.3
  canvas = rng.uniform(-1, 1, (2, Mh, Mw)).astype(np.float32)
  for red in _ordered.REDUCTIONS:
    values = rng.uniform(0.9, 1.1, (2, N)).astype(np.float32)
    check_against_shim(values, coords, valid, canvas, None, red, f"{red} {Mh}x{Mw}")


def test_mean_count_stops_at_2_pow_24():
  """torch_scatter's scatter_mean counts hits with float32 ones: 2^24 + 1 rounds back to 2^24, so a cell with more
  hits divides by 2^24.  2^24 + 5 hits of 2.0: the float32 sum stops at 2^25 (2^25 + 2 rounds to even), and the
  mean is 2^25 / 2^24 = 2.0 — not 2^25 / (2^24 + 5) = 1.9999995."""
  n = (1 << 24) + 5
  values = np.full((1, n), 2.0, np.float32)
  coords = np.zeros((1, n, 2), np.int64)
  canvas = np.zeros((1, 1, 1), np.float32)
  want = shim_scatter(values, coords, None, canvas, 0.0, "mean")[0]
  got, mask = orc.scatter(values, coords, None, canvas, 0.0, "mean")
  assert want.reshape(()) == np.float32(2.0)
  assert got.reshape(()) == want.reshape(()), (
    f"oracle {got.reshape(()).view(np.uint32):#010x} ({got.reshape(())!r}), "
    f"reference semantics {want.reshape(()).view(np.uint32):#010x} ({want.reshape(())!r})")
  assert mask.all()


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
def test_orth_project_ordered_matches_reference(red):
  """The restatement of the composed path against the reference's orth_project outputs in reduce.npz."""
  g = Golden("reduce")
  kw = g.kwargs
  fill = 1.0 if red == "prod" else 0.0
  top, mask, hgt = _ordered.orth_project_ordered(g["depth"], g["values"], None, g["pose"], 25., 0., np.float32(PITCH),
                                                 np.float32(0.88), fill_value=fill, reduction=red, **kw)
  assert_same(top, g[f"orth_top_{red}"], f"{red} topdown")
  assert_same(mask, g[f"orth_mask_{red}"], f"{red} mask")
  assert_same(hgt[:, :1], g[f"orth_height_{red}"], f"{red} height")


def test_orth_project_ordered_max_equals_the_oracle():
  """With max the restatement must give what the oracle's fused orth_project gives (every option switched on)."""
  for seed in range(6):
    depth, values, valid, pose, woff, hoff, pitch, camh, kw = _ordered.orth_case(7300 + seed)
    if depth.shape[1] != 1:
      continue
    kw = dict(kw, reduction=None, fill_value=kw["fill_value"] if kw["fill_value"] is not None else -np.inf)
    if "label_map" in kw:
      values = _ordered.one_hot(kw.pop("label_map"), kw.pop("num_classes"))
    want = orc.orth_project(depth, values, valid, pose, woff, hoff, pitch, camh, **kw)
    got = _ordered.orth_project_ordered(depth, values, valid, pose, woff, hoff, pitch, camh, **kw)
    for i, what in enumerate(("topdown", "mask", "height")[:len(want)]):
      w, o = want[i], got[i]
      assert_same(o[:, :w.shape[1]] if i == 2 else o, w, f"seed {seed} {what}")


def test_sum_bound_catches_a_lost_hit():
  rng = np.random.default_rng(5)
  values = rng.uniform(-1, 1, (2, 5000)).astype(np.float32)
  coords = np.stack((rng.integers(0, 3, (2, 5000)), rng.integers(0, 3, (2, 5000))), -1)
  canvas = np.zeros((2, 3, 3), np.float32)
  cv, _ = orc.scatter(values, coords, None, canvas, None, "sum")
  assert _ordered.sum_bound_violations(cv, values, coords, None, canvas) == 0
  lost = cv.copy()
  lost[1, 2, 0] -= values[1, np.flatnonzero((coords[1, :, 0] == 2) & (coords[1, :, 1] == 0))[0]]
  assert _ordered.sum_bound_violations(lost, values, coords, None, canvas) == 1
