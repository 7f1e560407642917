"""Reduction.sum / mean / prod on the GPU (csrc/dm_ordered.cu: key kernels, a stable radix sort, one thread folding
each cell's hits in the reference's point order) through every public entry that reaches it — project /
scatter_tensor, orth_project's composed path (value maps, label maps, the host entry), fuse_topdown_maps,
merge_into_canvas and MapBuilder — against the oracle (oracle/dm_oracle.c, pinned to the reference in
tests/test_ordered_oracle.py), bit for bit, at the sizes, key spaces and values where such kernels go wrong.
"""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import synth
from oracle import dm_oracle as orc
from tests import _ordered
from tests._golden import assert_same
from tests.test_gpu_parity import assert_workspaces_clean

pytestmark = pytest.mark.gpu

HFOV, PITCH = _ordered.HFOV, _ordered.PITCH


def npy(t):
  return t.detach().cpu().numpy()


def cu(a):
  return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(autouse=True)
def _device_clean():
  yield
  assert_workspaces_clean()


def gpu_project(values, coords, valid, canvas, fill, red, canvas_masks=None):
  """project() on device copies; also checks that the caller's canvas and values are left as they were."""
  v, c, cv = cu(values), cu(coords), cu(canvas)
  v0, cv0 = v.clone(), cv.clone()
  out = dmap.project(c, v, None if valid is None else cu(valid), cv,
                     canvas_masks=None if canvas_masks is None else cu(canvas_masks), fill_value=fill, reduction=red)
  assert torch.equal(v.nan_to_num(), v0.nan_to_num()) and torch.equal(cv.nan_to_num(), cv0.nan_to_num()), \
      "the caller's values or canvas were written"
  return npy(out[0]), npy(out[1])


def check_project(values, coords, valid, canvas, fill, red, what):
  want = orc.scatter(values, coords, valid, canvas, fill, red)
  got = gpu_project(values, coords, valid, canvas, fill, red)
  assert_same(got[0], want[0], f"{what} values")
  assert_same(got[1], want[1], f"{what} mask")
  if red == "sum":
    base = canvas if fill is None else np.full_like(canvas, fill)
    assert _ordered.sum_bound_violations(got[0], values, coords, valid, base) == 0, f"{what}: float64 bound"
  return got


# ---- a. project / scatter_tensor ----------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(30))
def test_project_random_vs_oracle(seed):
  values, coords, valid, canvas, fill, red = _ordered.scatter_case(9100 + seed, max_n=1_000_000 if seed % 5 == 0
                                                                   else 200_000)
  check_project(values, coords, valid, canvas, fill, red, f"seed {seed} {red} fill={fill}")


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
def test_project_heavy_collisions_and_sparse(red):
  """10^6 hits into 1x1 and 2x3 canvases (runs of 10^5..10^6 hits, one thread each); a 1000x1000 canvas with a few
  hundred points."""
  rng = np.random.default_rng(31)
  N = 1_000_000
  lo, hi = (0.9999, 1.0001) if red == "prod" else (-2.0, 2.0)
  for Mh, Mw, B in ((1, 1, 1), (2, 3, 2)):
    values = rng.uniform(lo, hi, (B, N // B)).astype(np.float32)
    coords = np.stack((rng.integers(0, Mh, (B, N // B)), rng.integers(0, Mw, (B, N // B))), -1)
    canvas = rng.uniform(-1, 1, (B, Mh, Mw)).astype(np.float32)
    for fill in (None, 1.0 if red == "prod" else 0.0):
      check_project(values, coords, None, canvas, fill, red, f"{red} {B}x{Mh}x{Mw} fill={fill}")
  values = rng.uniform(lo, hi, (2, 300)).astype(np.float32)
  coords = rng.integers(0, 1000, (2, 300, 2))
  coords[:, :40] = coords[:, :1]  # one cell with 40 hits among the scattered ones
  canvas = np.zeros((2, 1000, 1000), np.float32)
  check_project(values, coords, None, canvas, None, red, f"{red} sparse")


def _edge_case(total, seed):
  """(B, Mh, Mw) with B*Mh*Mw == total, and points that hit the first, middle and last cells of the key space over
  and over, interleaved with scattered ones."""
  rng = np.random.default_rng(seed)
  B = 2 if total % 2 == 0 and total > 2 else 1
  per = total // B
  Mh = next(d for d in (3, 2, 1) if per % d == 0)
  Mw = per // Mh
  M = Mh * Mw
  N = int(min(4 * M, 300_000)) + 64
  cell = rng.integers(0, M, (B, N))
  hot = np.asarray([0, 1, M // 2, max(M // 2 - 1, 0), M - 2, M - 1]) % M
  cell[:, ::5] = hot[rng.integers(0, hot.size, cell[:, ::5].shape)]
  coords = np.stack((cell // Mw, cell % Mw), -1)
  return B, Mh, Mw, coords


@pytest.mark.parametrize("k", [1, 8, 16, 20, 24])
def test_project_key_space_edges(k):
  """Key spaces of 2^k - 1, 2^k and 2^k + 1 cells: the sort examines only the significant key bits (bits_for), and
  dropped points carry the all-ones key that must sort after every real one."""
  for j, total in enumerate((2 ** k - 1, 2 ** k, 2 ** k + 1)):
    if total < 1:
      continue
    B, Mh, Mw, coords = _edge_case(total, 100 * k + j)
    N = coords.shape[1]
    rng = np.random.default_rng(k + j)
    for red in _ordered.REDUCTIONS:
      lo, hi = (0.99, 1.01) if red == "prod" else (-3.0, 3.0)
      values = rng.uniform(lo, hi, (B, N)).astype(np.float32)
      valid = rng.random((B, N)) > 0.1
      canvas = rng.uniform(-1, 1, (B, Mh, Mw)).astype(np.float32)
      check_project(values, coords, valid, canvas, None, red, f"{red} {B}x{Mh}x{Mw}")


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
def test_project_special_values_and_canvas_masks(red):
  rng = np.random.default_rng(41)
  Mh, Mw, N = 6, 7, 3000
  values = _ordered.special_values((2, 3, N), 42, 0.5, 1.5, rate=0.03)
  coords = np.stack((rng.integers(-1, Mh + 1, (2, 1, N)), rng.integers(-1, Mw + 1, (2, 1, N))), -1)
  valid = rng.random((2, 1, N)) > 0.2
  canvas = _ordered.special_values((2, 3, Mh, Mw), 43, -1.0, 1.0, rate=0.2)
  for fill in (None, 0.0, 1.0, -np.inf, np.nan, -0.0):
    check_project(values, coords, valid, canvas, fill, red, f"{red} fill={fill}")
  # +-x pairs that return exactly to the fill: hit, unchanged, mask False
  x = np.asarray([1.5, 0.25, 1e30], np.float32)
  pv = np.concatenate((x, -x))[None]
  pc = np.asarray([[[0, 0], [2, 3], [5, 6]] * 2])
  got = check_project(pv, pc, None, np.zeros((1, Mh, Mw), np.float32), 0.0, "sum", "cancelling pairs")
  assert not got[1].any()
  cm = rng.random((2, 3, Mh, Mw)) > 0.5
  want = orc.scatter(values, coords, valid, canvas, 0.0, red)
  got = gpu_project(values, coords, valid, canvas, 0.0, red, canvas_masks=cm)
  assert_same(got[0], want[0], "canvas_masks values")
  assert_same(got[1], want[1] | cm, "canvas_masks mask")


def test_scatter_tensor_broadcasting():
  """(N,) values and (N,) masks against a batched canvas and (B, N, 2) indices; (B, N) values against one (N, 2)
  index set."""
  rng = np.random.default_rng(51)
  B, N, Mh, Mw = 4, 5000, 9, 10
  canvas = rng.uniform(-1, 1, (B, Mh, Mw)).astype(np.float32)
  for red in _ordered.REDUCTIONS:
    v1 = rng.uniform(0.9, 1.1, (N,)).astype(np.float32)
    idx = rng.integers(-1, 11, (B, N, 2))
    m1 = rng.random(N) > 0.3
    got = dmap.utils.scatter_tensor(cu(canvas), cu(idx), cu(v1), masks=cu(m1), fill_value=None, reduction=red)
    want = orc.scatter(np.broadcast_to(v1, (B, N)), idx, np.broadcast_to(m1, (B, N)), canvas, None, red)
    assert_same(npy(got[0]), want[0], f"{red} (N,) values")
    assert_same(npy(got[1]), want[1], f"{red} (N,) values mask")
    vb = rng.uniform(0.9, 1.1, (B, N)).astype(np.float32)
    idx1 = rng.integers(0, 9, (N, 2))
    got = dmap.utils.scatter_tensor(cu(canvas), cu(idx1), cu(vb), fill_value=0.0, reduction=red)
    want = orc.scatter(vb, np.broadcast_to(idx1, (B, N, 2)), None, canvas, 0.0, red)
    assert_same(npy(got[0]), want[0], f"{red} one index set")
    assert_same(npy(got[1]), want[1], f"{red} one index set mask")


def _fold_loop(canvas, idx, values, valid, fill, red):
  """scatter_tensor on an n-D canvas, one float32 operation per hit in index order (utils.py:389-492)."""
  B = canvas.shape[0]
  dims = canvas.shape[1:]
  out = (np.full(canvas.shape, fill, np.float32) if fill is not None else canvas.copy()).reshape(B, -1)
  before = out.copy()
  cnt = np.zeros(out.shape, np.int64)
  for s in range(B):
    for i in range(values.shape[1]):
      ix = idx[s, i]
      if not valid[s, i] or any(x < 0 or x >= d for x, d in zip(ix, dims)):
        continue
      f = int(np.ravel_multi_index(tuple(ix), dims))
      out[s, f] = out[s, f] * values[s, i] if red == "prod" else out[s, f] + values[s, i]
      cnt[s, f] += 1
  if red == "mean":
    out = out / np.maximum(cnt, 1).astype(np.float32)
  with np.errstate(invalid="ignore"):
    mask = np.nan_to_num(np.abs(out - before)) != 0
  return out.reshape(canvas.shape), mask.reshape(canvas.shape)


@pytest.mark.parametrize("dims", [(37,), (4, 5, 6)])
def test_scatter_tensor_1d_and_3d_canvases(dims):
  """n = 1 and n = 3 (indices raveled into one row: utils.ravel_index) against a plain loop."""
  rng = np.random.default_rng(len(dims))
  B, N = 2, 700
  canvas = rng.uniform(-1, 1, (B,) + dims).astype(np.float32)
  idx = np.stack([rng.integers(-1, d + 1, (B, N)) for d in dims], -1)
  valid = rng.random((B, N)) > 0.2
  for red, fill in (("sum", None), ("mean", 0.0), ("prod", 1.0), ("sum", 0.0)):
    values = rng.uniform(0.8, 1.2, (B, N)).astype(np.float32)
    got = dmap.utils.scatter_tensor(cu(canvas), cu(idx), cu(values), masks=cu(valid), fill_value=fill, reduction=red)
    want = _fold_loop(canvas, idx, values, valid, fill, red)
    assert_same(npy(got[0]), want[0], f"{red} {dims}")
    assert_same(npy(got[1]), want[1], f"{red} {dims} mask")


# ---- b. the mean of a cell with more than 2^24 hits -----------------------------------------------------------------

def test_mean_count_stops_at_2_pow_24():
  """2^24 + 5 hits of 2.0 into one cell: torch_scatter's float32 count stops at 2^24, the sum at 2^25, so the
  mean is exactly 2.0 (the oracle's rule since it was fixed; tests/test_ordered_oracle.py pins it to the shim)."""
  n = (1 << 24) + 5
  values = np.full((1, n), 2.0, np.float32)
  coords = np.zeros((1, n, 2), np.int64)
  canvas = np.zeros((1, 1, 1), np.float32)
  for red, want in (("mean", 2.0), ("sum", 2.0 ** 25)):
    got, mask = gpu_project(values, coords, None, canvas, 0.0, red)
    oracle, _ = orc.scatter(values, coords, None, canvas, 0.0, red)
    g, w = got.reshape(()), np.float32(want)
    assert g == w and oracle.reshape(()) == w, (
      f"{red}: got {g.view(np.uint32):#010x} ({g!r}), want {w.view(np.uint32):#010x} ({w!r})")
    assert mask.all()


# ---- c. orth_project's composed path ------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(24))
def test_orth_project_composed_vs_oracle(seed):
  depth, values, valid, pose, woff, hoff, pitch, camh, kw = _ordered.orth_case(8200 + seed)
  want = _ordered.orth_project_ordered(depth, values, valid, pose, woff, hoff, pitch, camh, **kw)
  gkw = dict(kw)
  if "label_map" in gkw:
    gkw["label_map"] = cu(gkw["label_map"])
  got = dmap.orth_project(cu(depth), None if values is None else cu(values), None if valid is None else cu(valid), pose,
                          woff, hoff, pitch, camh, device="cuda", **gkw)
  assert len(got) == len(want)
  for g, w, what in zip(got, want, ("topdown", "mask", "height")):
    assert_same(npy(g), w, f"{kw['reduction']} {what}")


def test_orth_project_host_entry_composed():
  from dungeon_maps_b200 import hostapi
  for seed in range(40):
    depth, values, valid, pose, woff, hoff, pitch, camh, kw = _ordered.orth_case(8300 + seed)
    if values is not None and depth.shape[1] == 1:
      break
  want = _ordered.orth_project_ordered(depth, values, valid, pose, woff, hoff, pitch, camh, **kw)
  got = hostapi.orth_project_host(depth, values, valid, pose, woff, hoff, pitch, camh, **kw)
  for g, w, what in zip(got, want, ("topdown", "mask", "height")):
    assert_same(np.asarray(g), w, f"host {kw['reduction']} {what}")


# ---- d. full config 2 ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("red", ["sum", "mean"])
def test_orth_project_full_config2(red):
  """BASELINE config 2 (64 x 480x640 + 16 one-hot channels → 400x400, 314 M points through the sort): frames
  bit-exact against the oracle, two calls identical, and for sum every cell equals the integer count of its class
  hits (exact in float32 below 2^24, whatever the order)."""
  b, H, W, C = 64, 480, 640, 16
  depth, values, pose = synth.frames("room", b, H, W, C, seed=3, device="cuda")
  proj = dmap.MapProjector(width=W, height=H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=200., height_offset=0.,
                           cam_pitch=PITCH, cam_height=0.88, map_res=0.03, map_width=400, map_height=400,
                           trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=10, to_global=False,
                           fill_value=0.0, reduction=red)
  top, mask, hgt = proj.orth_project(depth, values, cam_pose=pose, get_height_map=True)
  top2, mask2, _ = proj.orth_project(depth, values, cam_pose=pose, get_height_map=True)
  assert torch.equal(top, top2) and torch.equal(mask, mask2), "two calls differ"
  k = proj.cam_params
  geo = (200., 0., PITCH, 0.88, 0.03, 400, 400, k.fx, k.fy, k.cx, k.cy, 0.15, 5.05, None, 10, False)
  sel = [0, 17, 63]
  want = _ordered.orth_project_ordered(npy(depth[sel]), npy(values[sel]), None, npy(pose[sel]), *geo, fill_value=0.0,
                                       reduction=red, get_height_map=True)
  assert_same(npy(top[sel]), want[0], "topdown slice")
  assert_same(npy(mask[sel]), want[1], "mask slice")
  assert_same(npy(hgt[sel]), want[2], "height slice")
  if red != "sum":
    return
  d, v, p = npy(depth), npy(values), npy(pose)
  top = npy(top)
  M = 400 * 400
  for f in range(b):
    coords, _, ok = _ordered.ordered_cells(d[f:f + 1], None, p[f:f + 1], 200., 0., PITCH, 0.88, 0.03, 400, k.fx, k.fy,
                                           k.cx, k.cy, 0.15, 5.05, None, 10, False)
    co, ok = coords[0, 0], ok[0, 0]
    inb = ok & (co[:, 0] >= 0) & (co[:, 0] < 400) & (co[:, 1] >= 0) & (co[:, 1] < 400)
    cell = (co[:, 0] * 400 + co[:, 1])[inb]
    hits = v[f].reshape(C, -1)[:, inb]
    for c in range(C):
      count = np.bincount(cell, weights=hits[c].astype(np.float64), minlength=M)
      assert (top[f, c].reshape(-1).astype(np.float64) == count).all(), f"frame {f} class {c}: sum != count"


# ---- e. fuse_topdown_maps -----------------------------------------------------------------------------------------

def _source(rng, b, C, h, w, res, to_global, pose, values):
  """A random top-down map: heights, a mask with about half the cells valid, values in [-2, 2) (or a height map)."""
  hgt = rng.uniform(-1, 2, (b, 1 if values else C, h, w)).astype(np.float32)
  mask = rng.random((b, C, h, w)) > 0.5
  vals = rng.uniform(-2, 2, (b, C, h, w)).astype(np.float32) if values else None
  woff, hoff = np.float32(w / 2 + rng.normal()), np.float32(rng.normal() + (h / 2 if to_global else 0))
  return dict(height=hgt, mask=mask, values=vals, woff=woff, hoff=hoff, res=res, to_global=to_global, pose=pose)


def _gpu_map(s, b_full=None, fill=0.0):
  C = s["mask"].shape[1]
  hgt = cu(s["height"])
  hgt = hgt.expand(-1, C, -1, -1) if s["values"] is not None else hgt
  top = hgt if s["values"] is None else cu(s["values"])
  proj = dmap.MapProjector(width=64, height=48, hfov=HFOV, cam_pose=s["pose"], width_offset=float(s["woff"]),
                           height_offset=float(s["hoff"]), map_res=s["res"], to_global=s["to_global"],
                           fill_value=fill)
  return dmap.TopdownMap(topdown_map=top, mask=cu(s["mask"]), height_map=hgt, map_projector=proj,
                         is_height_map=s["values"] is None)


def _oracle_source(s, b):
  C = s["mask"].shape[1]
  sh = (b,) + s["mask"].shape[1:]
  pose = np.ascontiguousarray(np.broadcast_to(np.asarray(s["pose"], np.float32).reshape(-1, 3), (b, 3)))
  return orc.FuseSource(np.broadcast_to(s["height"], sh), np.broadcast_to(s["mask"], sh),
                        None if s["values"] is None else np.broadcast_to(s["values"], sh), s["woff"], s["hoff"],
                        s["res"], True, s["to_global"], pose)


FUSE_CASES = [  # reduction, b, C (0: height maps), fill (None: the projector's -7), sources, global target, broadcast
  ("sum", 1, 0, 0.0, 2, True, False), ("mean", 3, 0, None, 3, False, False), ("prod", 4, 0, 1.0, 4, True, False),
  ("sum", 3, 2, None, 2, False, False), ("mean", 4, 2, 0.0, 3, True, False), ("prod", 1, 2, None, 4, False, False),
  ("sum", 4, 16, 0.0, 3, False, False), ("mean", 1, 16, -np.inf, 2, True, False), ("prod", 3, 16, np.nan, 3, False, False),
  ("sum", 4, 2, np.nan, 3, True, True), ("mean", 4, 0, 0.0, 2, False, True), ("prod", 4, 2, -np.inf, 4, True, True),
]


@pytest.mark.parametrize("case", range(len(FUSE_CASES)))
def test_fuse_topdown_maps_vs_oracle(case):
  """2 to 4 sources of different sizes and resolutions, local and global frames mixed, into a local or a global
  target; with `broadcast` the first source has batch 1 against the others' 4."""
  red, b, C, fill, n_src, target_global, broadcast = FUSE_CASES[case]
  rng = np.random.default_rng(600 + case)
  values = C > 0
  C = max(C, 1)
  srcs = []
  for i in range(n_src):
    h, w = int(rng.integers(5, 40)), int(rng.integers(5, 40))
    bs = 1 if (broadcast and i == 0) else b
    pose = synth.poses(bs, 700 + 10 * case + i, xz=0.6, yaw=1.0).numpy()
    srcs.append(_source(rng, bs, C, h, w, float(rng.choice([0.05, 0.1])), bool(i % 2), pose, values))
  tpose = synth.poses(b, 800 + case, xz=0.4, yaw=0.7).numpy()
  tgt = dmap.MapProjector(width=64, height=48, hfov=HFOV, cam_pose=tpose, map_res=0.05, to_global=target_global,
                          fill_value=-7.0, reduction=red)
  out = dmap.fuse_topdown_maps(*[_gpu_map(s) for s in srcs], map_projector=tgt, fill_value=fill)
  want = orc.fuse([_oracle_source(s, b) for s in srcs], target_global, tpose, 0.05, True, fill, -7.0, red)
  assert [out.proj.map_height, out.proj.map_width] == [want["map_height"], want["map_width"]], "shape"
  assert_same(np.asarray(out.proj.width_offset, np.float32).reshape(()), np.float32(want["width_offset"]), "woff")
  assert_same(np.asarray(out.proj.height_offset, np.float32).reshape(()), np.float32(want["height_offset"]), "hoff")
  assert_same(npy(out.topdown_map), want["topdown"], f"{red} fill={fill} topdown")
  assert_same(npy(out.mask), want["mask"], f"{red} fill={fill} mask")
  assert_same(npy(out.height_map), want["height"], f"{red} fill={fill} height")


# ---- f. merge_into_canvas and MapBuilder(fixed_canvas=...) ----------------------------------------------------------

def _still_source(b, C, Hc, Wc, res, values):
  """A global-frame map with the canvases' own geometry whose values (heights for a height map) are +0.0 and -0.0:
  a sum hits its cells and leaves every one of them as it was."""
  zero = np.where(np.arange(Wc) % 2 == 1, 0.0, -0.0).astype(np.float32)
  vals = np.broadcast_to(zero, (b, C, Hc, Wc)).copy()
  return dict(height=vals[:, :1] if values else vals, mask=np.ones((b, C, Hc, Wc), bool),
              values=vals if values else None, woff=np.float32(Wc / 2), hoff=np.float32(Hc / 2), res=res,
              to_global=True, pose=np.zeros((b, 3), np.float32))


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
@pytest.mark.parametrize("values", [False, True])
def test_merge_into_canvas_vs_oracle(red, values):
  """Four merges into the same canvases (b = 3), then one that adds zeros to every cell: for sum the cells keep their
  values and their mask bits, set or not."""
  rng = np.random.default_rng(61 + values)
  b, C, Hc, Wc, res = 3, (2 if values else 1), 37, 41, 0.05
  fill = 1.0 if red == "prod" else 0.0
  proj = dmap.MapProjector(width=64, height=48, hfov=HFOV, map_res=res, fill_value=fill, reduction=red)
  world, gw = None, None
  for t in range(5):
    if t < 4:
      s = _source(rng, b, C, int(rng.integers(10, 30)), int(rng.integers(10, 30)), res, bool(t % 2),
                  synth.poses(b, 900 + t, xz=0.5, yaw=1.0).numpy(), values)
    else:
      s = _still_source(b, C, Hc, Wc, res, values)
    world = orc.fuse_inplace(world, _oracle_source(s, b), (Hc, Wc), res, True, fill, red)
    gw = dmap.merge_into_canvas(gw, _gpu_map(s, fill=fill), (Hc, Wc), map_projector=proj)
    assert_same(npy(gw.topdown_map), world["topdown"], f"merge {t} topdown")
    assert_same(npy(gw.mask), world["mask"], f"merge {t} mask")
    if values:
      assert_same(npy(gw.height_map), world["height"], f"merge {t} height")
    if t == 3:
      before = (world["topdown"].copy(), world["mask"].copy())
  if red == "sum":  # the last merge hit every cell and changed none of them
    assert_same(world["topdown"], before[0], "zero merge values")
    assert_same(world["mask"], before[1], "zero merge mask")
    assert before[1].any() and not before[1].all()


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
def test_fixed_canvas_builder_vs_oracle(red):
  b, H, W = 3, 60, 80
  fill = 1.0 if red == "prod" else 0.0
  proj = dmap.MapProjector(width=W, height=H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=0., height_offset=0.,
                           cam_pitch=PITCH, cam_height=0.88, map_res=0.05, map_width=60, map_height=60,
                           trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=2, to_global=True,
                           fill_value=fill, reduction=red, device="cuda")
  builder = dmap.MapBuilder(map_projector=proj, fixed_canvas=(71, 67))
  k = proj.cam_params
  world, pose = None, torch.zeros(b, 3)
  for t in range(4):
    pose = pose + synth.poses(b, 70 + t, xz=0.5, yaw=0.8)
    depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, pose, seed=7)
    builder.step(depth_map=depth, cam_pose=pose, to_global=False, width_offset=30., height_offset=0.)
    top, mask, hgt = _ordered.orth_project_ordered(depth.numpy(), None, None, pose.numpy(), 30., 0., PITCH, 0.88, 0.05,
                                                   60, 60, k.fx, k.fy, k.cx, k.cy, 0.15, 5.05, None, 2, False, True,
                                                   fill, red, True)
    src = orc.FuseSource(hgt, mask, None, 30., 0., 0.05, True, False, pose.numpy())
    world = orc.fuse_inplace(world, src, (71, 67), 0.05, True, fill, red)
    assert_same(npy(builder.world_map.topdown_map), world["topdown"], f"step {t} topdown")
    assert_same(npy(builder.world_map.mask), world["mask"], f"step {t} mask")
  assert 0 < int(world["mask"].sum()) < world["mask"].size


# ---- g. MapBuilder's general path ---------------------------------------------------------------------------------

def _builder_run(red, C, to_global, b, H, W, T, M, res, seed):
  fill = 1.0 if red == "prod" else 0.0
  proj = dmap.MapProjector(width=W, height=H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=0., height_offset=0.,
                           cam_pitch=PITCH, cam_height=0.88, map_res=res, map_width=M, map_height=M,
                           trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=3, fill_value=fill,
                           to_global=to_global, reduction=red, device="cuda")
  k = proj.cam_params
  builder = dmap.MapBuilder(map_projector=proj)
  import sys
  sys.path.insert(0, str(__import__("pathlib").Path(__file__).resolve().parents[1]))
  from bench import BuilderWorkload
  poses = BuilderWorkload.walk(b, T, seed=seed, half=M * res / 3)
  world = None
  for t in range(T):
    depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t], seed=seed, half=M * res / 2)
    vals = None if C == 0 else synth.uniform((b, C, H, W), seed + t, 0.5, 1.5)
    local = builder.step(depth, value_map=vals, cam_pose=poses[t], to_global=False, width_offset=M / 2.,
                         height_offset=0., map_width=M, map_height=M)
    p = poses[t].numpy()
    lt, lm, lh = _ordered.orth_project_ordered(depth.numpy(), None if vals is None else vals.numpy(), None, p, M / 2., 0.,
                                               PITCH, 0.88, res, M, M, k.fx, k.fy, k.cx, k.cy, 0.15, 5.05, None, 3,
                                               False, True, fill, red, True)
    assert_same(npy(local.topdown_map), lt, f"step {t} local topdown")
    assert_same(npy(local.mask), lm, f"step {t} local mask")
    src = [orc.FuseSource(lh, lm, None if C == 0 else lt, M / 2., 0., res, True, False, p)]
    if world is not None:
      src.insert(0, orc.FuseSource(world["height"], world["mask"], None if C == 0 else world["topdown"],
                                   world["width_offset"], world["height_offset"], res, True, to_global, poses[t - 1].numpy()))
    world = orc.fuse(src, to_global, p, res, True, None, fill, red)
    wm = builder.world_map
    assert [wm.proj.map_height, wm.proj.map_width] == [world["map_height"], world["map_width"]], f"step {t} shape"
    assert_same(np.asarray(wm.proj.width_offset, np.float32).reshape(()), np.float32(world["width_offset"]), "woff")
    assert_same(np.asarray(wm.proj.height_offset, np.float32).reshape(()), np.float32(world["height_offset"]), "hoff")
    assert_same(npy(wm.topdown_map), world["topdown"], f"step {t} world topdown")
    assert_same(npy(wm.mask), world["mask"], f"step {t} world mask")
    assert_same(npy(wm.height_map), world["height"], f"step {t} world height")


@pytest.mark.parametrize("red", _ordered.REDUCTIONS)
@pytest.mark.parametrize("C,to_global", [(0, True), (2, False)])
def test_map_builder_general_path_vs_oracle(red, C, to_global):
  _builder_run(red, C, to_global, b=4, H=60, W=80, T=4, M=60, res=0.1, seed=11)


def test_map_builder_config4_shapes_sum():
  _builder_run("sum", 0, True, b=4, H=480, W=640, T=4, M=400, res=0.03, seed=2)


# ---- h. a side stream ---------------------------------------------------------------------------------------------

def test_side_stream_equals_default_stream():
  """Inputs produced on a side stream and the call made there give the default stream's results (the scratch comes
  from the stream-ordered allocator of the caller's stream)."""
  values, coords, valid, canvas, fill, _ = _ordered.scatter_case(77, max_n=400_000)
  rng = np.random.default_rng(78)
  srcs = [_source(rng, 3, 2, 30, 20, 0.05, bool(i), synth.poses(3, 79 + i).numpy(), True) for i in range(2)]
  tgt = dmap.MapProjector(width=64, height=48, hfov=HFOV, map_res=0.05, to_global=True, fill_value=0.0, reduction="sum")

  def run():
    a = dmap.project(cu(coords) + 0, cu(values) * 1.0, None if valid is None else cu(valid), cu(canvas) * 1.0,
                     fill_value=fill, reduction="sum")
    f = dmap.fuse_topdown_maps(*[_gpu_map(s) for s in srcs], map_projector=tgt)
    m = dmap.merge_into_canvas(None, _gpu_map(srcs[0]), (45, 51), map_projector=tgt)
    m = dmap.merge_into_canvas(m, _gpu_map(srcs[1]), (45, 51), map_projector=tgt)
    return [a[0], a[1], f.topdown_map, f.mask, f.height_map, m.topdown_map, m.mask, m.height_map]

  want = [t.clone() for t in run()]
  torch.cuda.synchronize()
  side = torch.cuda.Stream()
  with torch.cuda.stream(side):
    got = run()
  side.synchronize()
  for i, (w, g) in enumerate(zip(want, got)):
    assert torch.equal(w.nan_to_num(), g.nan_to_num()) and torch.equal(w.isnan(), g.isnan()), f"output {i} differs"
