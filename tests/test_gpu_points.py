"""The point primitives of csrc/dm_points.cu through their public entries — utils.rotate / translate, the four space
transforms, image_to_camera_space / camera_to_image_space, depth_map_to_point_cloud, map_quantize / map_dequantize /
height_map_to_point_cloud, crop_topdown_map / TopdownMap.select and TopdownMap.get_coords / get_points / get_camera /
get_origin — against the oracle (oracle/dm_oracle.c, pinned to the reference in tests/test_oracle_golden.py), bit for
bit, where these kernels could go wrong: batches with distinct parameters per sample, 4-point groups that straddle
samples and frames, sizes that take several passes of the grid-stride loop, unaligned inputs that take the scalar
paths, and NaN / inf / out-of-range / tie values.  The oracle indexes with plain nested loops, so none of the kernels'
flat, grouped or strided index arithmetic is shared with it."""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from oracle import dm_oracle as orc
from tests._golden import assert_same

pytestmark = pytest.mark.gpu

INT64_MIN = np.iinfo(np.int64).min
SPECIALS = np.float32([np.nan, np.inf, -np.inf, 0.0, -0.0, 1e30, -1e30])


def npy(t):
  return t.detach().cpu().numpy()


def cu(a):
  return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def unaligned(a, k):
  """A contiguous CUDA copy of `a` that starts k elements into its allocation (not 16-byte aligned for k = 1..3)."""
  t = torch.from_numpy(np.ascontiguousarray(a))
  v = torch.empty(t.numel() + k, dtype=t.dtype, device="cuda")[k:].view(t.shape)
  v.copy_(t)
  assert v.is_contiguous() and v.data_ptr() % 16 != 0
  return v


def twice(fn):
  """fn() as numpy (a tuple for several results), after checking that a second call gives identical bits."""
  def run():
    out = fn()
    return tuple(npy(o) for o in out) if isinstance(out, tuple) else npy(out)
  a, b = run(), run()
  for x, y in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
    assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), "a repeated call differs"
  return a


def pass_items(per_thread):
  """Items one pass of a point kernel's grid-stride loop covers: grid_for caps a launch at SMs x 16 blocks of 256."""
  return torch.cuda.get_device_properties(0).multi_processor_count * 16 * 256 * per_thread


def salted(shape, seed, lo=-8.0, hi=8.0):
  """Uniform float32 values with NaN, +-inf, +-0 and +-1e30 salted in."""
  rng = np.random.default_rng(seed)
  a = rng.uniform(lo, hi, shape).astype(np.float32)
  flat = a.reshape(-1)
  for k, v in enumerate(SPECIALS):
    flat[k::13] = v
  return a


def poses(b, seed):
  """(b, 3) [x, z, yaw], distinct per sample; one yaw inside the |yaw| <= 0.001 clamp."""
  rng = np.random.default_rng(seed)
  p = np.stack((rng.uniform(-5, 5, b), rng.uniform(-5, 5, b), rng.uniform(-math.pi, math.pi, b)), 1).astype(np.float32)
  p[-1, 2] = 0.0007
  return p


def pitch_height(b, seed):
  rng = np.random.default_rng(seed)
  return rng.uniform(-0.6, 0.3, b).astype(np.float32), rng.uniform(0.4, 1.6, b).astype(np.float32)


# ---- a. transforms ------------------------------------------------------------------------------------------------

def _space_cases(b, seed):
  """(name, gpu call, oracle step builder) of the four space transforms with per-sample parameters."""
  pose = poses(b, seed)
  pitch, camh = pitch_height(b, seed + 1)
  return [
    ("camera_to_local", lambda p: dmap.camera_to_local_space(p, pitch, camh),
     lambda n: orc.to_local_steps(pitch, camh, n)),
    ("local_to_camera", lambda p: dmap.local_to_camera_space(p, pitch, camh),
     lambda n: orc.to_camera_steps(pitch, camh, n)),
    ("local_to_global", lambda p: dmap.local_to_global_space(p, pose), lambda n: orc.to_global_steps(pose, n)),
    ("global_to_local", lambda p: dmap.global_to_local_space(p, pose), lambda n: orc.from_global_steps(pose, n)),
  ]


def _rot_steps(axis, ang, n):
  R = orc.rodrigues(axis, ang)
  return orc.steps(4, R, np.zeros((R.shape[0], 3), np.float32), n)


def _add_steps(off, n):
  off = np.asarray(off, np.float32).reshape(-1, 3)
  return orc.steps(3, np.zeros((off.shape[0], 9), np.float32), off, n)


@pytest.mark.parametrize("b", [3, 5])
@pytest.mark.parametrize("n", [1, 7, 44, 45, 1001])
def test_transforms_per_sample(b, n):
  """Every sample has its own parameters and n is not a multiple of 4, so 4-point groups straddle samples; 44 and 45
  sit on either side of the reference's switch to the fused (FMA) product."""
  pts = salted((b, n, 3), 100 * b + n)
  rng = np.random.default_rng(n)
  ang = rng.uniform(-3, 3, b).astype(np.float32)
  ang[0] = -0.0009
  axis = [0.3, -1.2, 0.5]
  off = rng.uniform(-4, 4, (b, 3)).astype(np.float32)
  cases = _space_cases(b, 7 * n + b) + [
    ("rotate", lambda p: dmap.utils.rotate(p, axis, ang), lambda k: _rot_steps(axis, ang, k)),
    ("rotate x", lambda p: dmap.utils.rotate(p, [1., 0., 0.], ang), lambda k: _rot_steps([1., 0., 0.], ang, k)),
    ("translate", lambda p: dmap.utils.translate(p, off), lambda k: _add_steps(off, k)),
  ]
  for name, gpu, steps in cases:
    got = twice(lambda: gpu(cu(pts)))
    assert_same(got, orc.transform_points(pts, [steps(n)]), f"{name} b={b} n={n}")


def test_transforms_5d_points():
  """(b, c, h, w, 3) points: the per-sample count is c * h * w (naive below 400 / 9, fused above)."""
  for shape in ((3, 2, 3, 5, 3), (4, 2, 5, 7, 3)):
    b, n = shape[0], int(np.prod(shape[1:-1]))
    pts = salted(shape, n)
    for name, gpu, steps in _space_cases(b, n):
      got = twice(lambda: gpu(cu(pts)))
      assert got.shape == shape
      want = orc.transform_points(pts.reshape(b, n, 3), [steps(n)]).reshape(shape)
      assert_same(got, want, f"{name} {shape}")


def test_transforms_broadcast():
  b, n = 4, 45
  pose = poses(b, 3)
  pitch, camh = pitch_height(b, 4)
  one = salted((1, n, 3), 5)
  many = salted((b, n, 3), 6)
  rep = np.ascontiguousarray(np.broadcast_to(one, (b, n, 3)))
  # one point set over b poses (get_camera's form)
  for name, gpu, steps in _space_cases(b, 8):
    assert_same(twice(lambda: gpu(cu(one))), orc.transform_points(rep, [steps(n)]), f"{name}: one set over b")
  # a single (3,) point over b poses: one point per sample (naive product)
  p3 = np.float32([0.75, -1.25, 2.5])
  got = twice(lambda: dmap.local_to_global_space(cu(p3), pose))
  assert_same(got, orc.transform_points(np.tile(p3, (b, 1, 1)), [orc.to_global_steps(pose, 1)]), "(3,) over b poses")
  # (n, 3) points are n samples of one point each; with b != n poses that is an error, as in the reference
  p2 = salted((b, 3), 9)
  got = twice(lambda: dmap.local_to_global_space(cu(p2), pose))
  assert_same(got, orc.transform_points(p2.reshape(b, 1, 3), [orc.to_global_steps(pose, 1)]).reshape(b, 3),
              "(b, 3) = one point per sample")
  with pytest.raises(ValueError):
    dmap.local_to_global_space(cu(salted((7, 3), 10)), pose)
  # one pose (and one pitch / height) over b point sets
  for p_one in (pose[1], pose[1:2]):
    got = twice(lambda: dmap.local_to_global_space(cu(many), p_one))
    want = orc.transform_points(many, [orc.to_global_steps(np.repeat(pose[1:2], b, 0), n)])
    assert_same(got, want, f"one pose {p_one.shape} over b sets")
  got = twice(lambda: dmap.camera_to_local_space(cu(many), float(pitch[2]), float(camh[2])))
  want = orc.transform_points(many, [orc.to_local_steps(np.repeat(pitch[2:3], b), np.repeat(camh[2:3], b), n)])
  assert_same(got, want, "one pitch / height over b sets")
  # rotate: one axis per sample (b calls of the oracle at batch 1), and one angle for the whole batch
  axes = np.float32([[1, 0, 0], [0.3, -1.2, 0.5], [0, 0, 1], [-2, 1, 0.25]])
  ang = np.float32([0.4, -2.9, 0.0005, 1.7])
  got = twice(lambda: dmap.utils.rotate(cu(many), axes, ang))
  want = np.concatenate([orc.transform_points(many[i:i + 1], [_rot_steps(axes[i].tolist(), ang[i:i + 1], n)])
                         for i in range(b)])
  assert_same(got, want, "rotate with one axis per sample")
  got = twice(lambda: dmap.utils.rotate(cu(many), [0., 1., 0.], 1.3))
  assert_same(got, orc.transform_points(many, [_rot_steps([0., 1., 0.], np.full(b, 1.3, np.float32), n)]),
              "rotate with one angle")
  got = twice(lambda: dmap.utils.translate(cu(many), [0.5, -2.0, 3.25]))
  assert_same(got, orc.transform_points(many, [_add_steps(np.tile([0.5, -2.0, 3.25], (b, 1)), n)]),
              "translate with one offset")


def test_step_cache_keys_the_fused_flag():
  """Interleaved calls that share their parameter bytes but not the fused flag, and the converse."""
  b = 3
  A, B = poses(b, 21), poses(b, 22)
  for k, (pose, n) in enumerate(((A, 44), (A, 45), (B, 44), (A, 44), (B, 45), (A, 45))):
    pts = salted((b, n, 3), 30 + k)
    want = orc.transform_points(pts, [orc.to_global_steps(pose, n)])
    other = orc.transform_points(pts, [orc.to_global_steps(pose, 89 - n)])
    assert not np.array_equal(want, other, equal_nan=True), "the fused flag must matter for these points"
    assert_same(twice(lambda: dmap.local_to_global_space(cu(pts), pose)), want, f"call {k} n={n}")


def test_transform_entry_with_three_steps_per_sample():
  """dm_transform_points_f32 with n_steps = 3 and distinct steps per sample: steps[s * n_steps + k]."""
  b, n = 5, 45
  pts = salted((b, n, 3), 40)
  pitch, camh = pitch_height(b, 41)
  st = np.ascontiguousarray(np.stack([orc.to_local_steps(pitch, camh, n), orc.to_global_steps(poses(b, 42), n),
                                      orc.from_global_steps(poses(b, 43), n)], axis=1))
  dev = torch.device("cuda", torch.cuda.current_device())
  steps = cu(st.view(np.uint8))

  def run():
    p = cu(pts)
    out = torch.empty_like(p)
    nat.check(nat.lib().dm_transform_points_f32(p.data_ptr(), steps.data_ptr(), 3, b, n, out.data_ptr(),
                                                nat.stream_ptr(dev)), "dm_transform_points_f32")
    return out
  assert_same(twice(run), orc.transform_points(pts, list(st.T)), "three steps per sample")


def test_transforms_multi_pass():
  b = 4
  bound = 3 * pass_items(4)
  n = bound // b + 7
  assert b * n >= bound and n % 4 != 0
  pts = salted((b, n, 3), 50)
  pose = poses(b, 51)
  got = twice(lambda: dmap.local_to_global_space(cu(pts), pose))
  assert_same(got, orc.transform_points(pts, [orc.to_global_steps(pose, n)]), "multi-pass local_to_global")


# ---- b. depth_map_to_point_cloud ----------------------------------------------------------------------------------

TMIN, TMAX = 0.5, 5.0


def depth_frames(shape, seed):
  rng = np.random.default_rng(seed)
  d = rng.uniform(0.1, 10.0, shape).astype(np.float32)
  flat = d.reshape(-1)
  for k, v in enumerate((TMIN, TMAX, np.nan, np.inf, -np.inf, 0.0, -1.5)):
    flat[k::11] = v
  return d


def _check_depth(depth, valid, vcu, what, trunc=((None, None), (TMIN, None), (None, TMAX), (TMIN, TMAX))):
  b, c, H, W = depth.shape
  k = orc.intrinsics(W, H, math.radians(70))
  for flip in (True, False):
    for tmin, tmax in trunc:
      got = twice(lambda: dmap.depth_map_to_point_cloud(depth if torch.is_tensor(depth) else cu(depth), vcu,
                                                        k["fx"], k["fy"], k["cx"], k["cy"], tmin, tmax, flip_h=flip))
      want = orc.depth_to_points(npy(depth) if torch.is_tensor(depth) else depth, valid, k["fx"], k["fy"], k["cx"],
                                 k["cy"], flip, tmin, tmax)
      tag = f"{what} flip={flip} tmin={tmin} tmax={tmax}"
      assert_same(got[0], want[0], f"{tag} points")
      assert_same(got[1], want[1], f"{tag} valid")
  return got


@pytest.mark.parametrize("shape", [(2, 3, 7, 9), (3, 1, 5, 5), (1, 2, 1, 13), (4, 1, 33, 17)])
def test_depth_to_points_groups_cross_frames(shape):
  b, c, H, W = shape
  assert (H * W) % 4 != 0
  depth = depth_frames(shape, sum(shape))
  rng = np.random.default_rng(H * W)
  full = rng.random(shape) > 0.3
  hw = rng.random((H, W)) > 0.3
  per_b = rng.random((b, 1, H, W)) > 0.3
  for valid in (None, full, hw, per_b):
    _check_depth(depth, valid, None if valid is None else cu(valid), f"{shape} valid {np.shape(valid)}")


def test_depth_to_points_multi_pass():
  H, W = 480, 640
  bound = 3 * pass_items(4)
  frames = -(-bound // (H * W))
  assert frames * H * W >= bound
  depth = depth_frames((frames, 1, H, W), 60)
  valid = np.random.default_rng(61).random((frames, 1, H, W)) > 0.2
  _check_depth(depth, valid, cu(valid), f"{frames}x480x640", trunc=((TMIN, TMAX),))


# ---- c. image_to_camera_space / camera_to_image_space -------------------------------------------------------------

def _image_points(shape, seed):
  p = salted(shape, seed, -50.0, 50.0)
  flat = p.reshape(-1, 3)
  flat[1::5, 2] = 0.0
  flat[2::5, 2] = np.float32(-1e-7)   # z + 1e-7 == 0
  flat[3::5, 2] = np.abs(flat[3::5, 2]) + 0.1
  return p


@pytest.mark.parametrize("flip", [True, False])
def test_image_camera(flip):
  k = dict(focal_x=23.5, focal_y=19.25, center_x=16.0, center_y=12.5)
  args = (k["focal_x"], k["focal_y"], k["center_x"], k["center_y"], flip)
  for shape, height in (((3, 5, 7, 3), None), ((2, 11, 13, 3), None), ((45, 3), 37), ((7, 3), 5)):
    pts = _image_points(shape, sum(shape))
    h = shape[-3] if height is None else height
    for to_image, fn in ((0, dmap.image_to_camera_space), (1, dmap.camera_to_image_space)):
      got = twice(lambda: fn(cu(pts), **k, flip_h=flip, height=height))
      assert_same(got, orc.image_camera(pts, *args, h, to_image), f"{fn.__name__} {shape} height={height}")


# ---- d. map_quantize / map_dequantize / height_map_to_point_cloud -------------------------------------------------

WOFF = np.float32([12.25, -3.5, 100.75, 0.0, 7.5])
HOFF = np.float32([-2.0, 40.25, 5.5, -60.75, 1.0])
MH = 64


def tie_values(off, res, count, seed):
  """float32 x with fl(fl(x / res) + off) == m + 0.5 exactly: floor(. + 0.5) rounds it half up to m + 1 (and with
  flip_h, (MH - 1) - (m + 0.5) is a tie too)."""
  rng = np.random.default_rng(seed)
  out = []
  for m in rng.integers(-300, 300, 50 * count):
    t = np.float32(m + 0.5) - np.float32(off)
    x = np.float32(float(t) * float(res))
    for _ in range(8):
      if np.float32(x / np.float32(res)) + np.float32(off) == np.float32(m + 0.5):
        out.append(x)
        break
      x = np.nextafter(x, np.float32(np.inf) if np.float32(x / np.float32(res)) < t else np.float32(-np.inf))
    if len(out) == count:
      return np.float32(out)
  raise AssertionError(f"no ties for offset {off} at res {res}")


BIG = np.float32([np.nan, np.inf, -np.inf, 3e19, -3e19, 1e18, -1e18, -0.0])


def quantize_inputs(b, per, woff, hoff, res, seed):
  """(b, per) x and z: uniform values, then per sample 6 ties, then the out-of-range / in-range / -0 values."""
  rng = np.random.default_rng(seed)
  x = rng.uniform(-20, 20, (b, per)).astype(np.float32)
  z = rng.uniform(-20, 20, (b, per)).astype(np.float32)
  for s in range(b):
    x[s, 3:9] = tie_values(woff[s], res, 6, seed + s)
    z[s, 11:17] = tie_values(hoff[s], res, 6, seed + 100 + s)
    x[s, 20:28] = BIG
    z[s, 30:38] = BIG
  return x, z


def _offset_forms(b):
  """(gpu argument, per-sample oracle values) of the offset forms: Python scalar, (1,), (b,) and (b, 1)."""
  w, h = WOFF[:b], HOFF[:b]
  return [(float(w[1]), float(h[1]), np.repeat(w[1], b), np.repeat(h[1], b)),
          (w[2:3].copy(), h[2:3].copy(), np.repeat(w[2], b), np.repeat(h[2], b)),
          (w.copy(), h.copy(), w, h),
          (torch.from_numpy(w.reshape(b, 1).copy()), torch.from_numpy(h.reshape(b, 1).copy()), w, h)]


def _check_quantize(x, z, woff, hoff, ow, oh, res, flip, what):
  b = x.shape[0] if x.ndim > 1 else 1
  xb2, zb2 = x.reshape(b, -1), z.reshape(b, -1)
  got = twice(lambda: dmap.map_quantize(cu(x), cu(z), woff, hoff, res, MH, flip_h=flip))
  out_shape = x.shape if x.ndim > 1 else (1, x.size)
  want = tuple(a.reshape(out_shape) for a in orc.map_quantize(xb2, zb2, ow, oh, res, MH, flip))
  assert got[0].dtype == np.int64
  assert_same(got[0], want[0], f"{what} x bins")
  assert_same(got[1], want[1], f"{what} z bins")
  return want


@pytest.mark.parametrize("res", [0.25, 0.05])
@pytest.mark.parametrize("flip", [True, False])
def test_map_quantize(res, flip):
  b, per = 4, 45
  for form, (woff, hoff, ow, oh) in enumerate(_offset_forms(b)):
    x, z = quantize_inputs(b, per, ow, oh, res, 70 + form)
    for shape in ((b, per), (b, 3, per // 3)):
      want = _check_quantize(x.reshape(shape), z.reshape(shape), woff, hoff, ow, oh, res, flip, f"{shape} form {form}")
      xw, zw = want[0].reshape(b, per), want[1].reshape(b, per)
      # the oracle's own bins show what the inputs exercise: ties round half up, the big values
      for s in range(b):
        ties = np.floor(x[s, 3:9] / np.float32(res) + ow[s]).astype(np.int64) + 1
        assert np.array_equal(xw[s, 3:9], ties)
        assert (xw[s, 20:25] == INT64_MIN).all() and (zw[s, 30:35] == INT64_MIN).all()
        if res == 0.25:
          assert (xw[s, 25:27] != INT64_MIN).all() and (zw[s, 35:37] != INT64_MIN).all()
  # (n,) coordinates: one sample
  x, z = quantize_inputs(1, 77, WOFF[3:4], HOFF[3:4], res, 79)
  for woff, hoff in ((float(WOFF[3]), float(HOFF[3])), (WOFF[3:4], HOFF[3:4])):
    _check_quantize(x[0], z[0], woff, hoff, WOFF[3:4], HOFF[3:4], res, flip, "(n,)")


@pytest.mark.parametrize("flip", [True, False])
def test_map_dequantize(flip):
  b, per, res = 4, 45, 0.05
  rng = np.random.default_rng(80)
  xb = rng.integers(-500, 500, (b, per))
  zb = rng.integers(-500, 500, (b, per))
  big = np.int64([(1 << 24) + 1, (1 << 30) + 3, -(1 << 25) - 1, (1 << 40) + 12345, -7, -(1 << 24) - 3])
  xb[:, 5:11] = big
  zb[:, 13:19] = big[::-1]
  for form, (woff, hoff, ow, oh) in enumerate(_offset_forms(b)):
    for shape in ((b, per), (b, 5, per // 5)):
      got = twice(lambda: dmap.map_dequantize(cu(xb.reshape(shape)), cu(zb.reshape(shape)), woff, hoff, res, MH,
                                              flip_h=flip))
      want = orc.map_dequantize(xb, zb, ow, oh, res, MH, flip)
      assert_same(got[0], want[0].reshape(shape), f"{shape} form {form} x")
      assert_same(got[1], want[1].reshape(shape), f"{shape} form {form} z")
  got = twice(lambda: dmap.map_dequantize(cu(xb[0]), cu(zb[0]), float(WOFF[2]), float(HOFF[2]), res, MH, flip_h=flip))
  want = orc.map_dequantize(xb[:1], zb[:1], WOFF[2:3], HOFF[2:3], res, MH, flip)
  assert_same(got[0], want[0], "(n,) x")
  assert_same(got[1], want[1], "(n,) z")


def test_map_quantize_multi_pass():
  b, res = 4, 0.05
  bound = 3 * pass_items(1)
  per = bound // b + 5
  assert b * per >= bound
  x, z = quantize_inputs(b, per, WOFF, HOFF, res, 90)
  xq = twice(lambda: dmap.map_quantize(cu(x), cu(z), WOFF[:b], HOFF[:b], res, MH, flip_h=True))
  want = orc.map_quantize(x, z, WOFF[:b], HOFF[:b], res, MH, True)
  assert_same(xq[0], want[0], "multi-pass x bins")
  assert_same(xq[1], want[1], "multi-pass z bins")
  xb = np.clip(want[0], -1 << 30, 1 << 30)
  zb = np.clip(want[1], -1 << 30, 1 << 30)
  got = twice(lambda: dmap.map_dequantize(cu(xb), cu(zb), WOFF[:b], HOFF[:b], res, MH, flip_h=False))
  wd = orc.map_dequantize(xb, zb, WOFF[:b], HOFF[:b], res, MH, False)
  assert_same(got[0], wd[0], "multi-pass dequantize x")
  assert_same(got[1], wd[1], "multi-pass dequantize z")


@pytest.mark.parametrize("flip", [True, False])
def test_height_map_to_point_cloud(flip):
  b, c, h, w = 3, 2, 10, 12
  hm = salted((b, c, h, w), 95)
  res = 0.1
  got = twice(lambda: dmap.height_map_to_point_cloud(cu(hm), WOFF[:b], HOFF[:b], res, h, flip_h=flip))
  r, cc = np.divmod(np.arange(c * h * w) % (h * w), w)
  cols = np.tile(cc.astype(np.float32), (b, 1))
  rows = np.tile(r.astype(np.float32), (b, 1))
  x, z = orc.map_dequantize(cols, rows, WOFF[:b], HOFF[:b], res, h, flip)
  want = np.stack((x.reshape(b, c, h, w), hm, z.reshape(b, c, h, w)), -1)
  assert_same(got, want, "height_map_to_point_cloud")


# ---- e. crop_topdown_map / TopdownMap.select ----------------------------------------------------------------------

def _crop_source(b, C, h, w, seed, fill_value, stride0=False, woff=None, hoff=None, flip=True):
  rng = np.random.default_rng(seed)
  top = salted((b, C, h, w), seed)
  mask = rng.random((b, C, h, w)) > 0.4
  hm1 = rng.uniform(-1, 2, (b, 1 if stride0 else C, h, w)).astype(np.float32)
  hm_t = cu(hm1)
  if stride0:
    hm_t = hm_t.expand(b, C, h, w)
  proj = dmap.MapProjector(width=16, height=12, hfov=1.2, map_res=0.05, map_width=w, map_height=h,
                           width_offset=WOFF[:b].copy() if woff is None else woff,
                           height_offset=HOFF[:b].copy() if hoff is None else hoff, flip_h=flip, fill_value=fill_value)
  src = dmap.TopdownMap(topdown_map=cu(top), mask=cu(mask), height_map=hm_t, map_projector=proj)
  return src, top, mask, hm1


def _check_crop(src, top, mask, hm1, center, cw, ch, fill_value, what):
  b, C = top.shape[:2]
  out = twice(lambda: (lambda m: (m.topdown_map, m.mask, m.height_map))(src.select(center, cw, ch)))
  assert_same(out[0], orc.crop_nearest(top, center, cw, ch, fill_value), f"{what} values")
  want_mask = orc.crop_nearest(mask.astype(np.float32), center, cw, ch, 0.0) != 0
  assert out[1].dtype == np.bool_
  assert_same(out[1], want_mask, f"{what} mask")
  want_h = np.broadcast_to(orc.crop_nearest(hm1, center, cw, ch, -np.inf), (b, C, ch, cw))
  assert_same(out[2], want_h, f"{what} height")


CENTERS = np.float32([[5.0, 4.0],        # inside
                      [0.0, 10.0],       # on the edge
                      [-3.0, -6.5],      # negative, outside
                      [30.0, 2.5],       # outside, .5
                      [6.5, 3.5]])       # .5 ties


@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("fill_value", [None, -7.0])
def test_select(C, fill_value):
  b, h, w = 3, 11, 13
  for k, (cw, ch) in enumerate(((7, 5), (6, 4), (1, 1), (25, 20))):
    for stride0 in (False, True):
      src, top, mask, hm1 = _crop_source(b, C, h, w, 100 + k, fill_value, stride0)
      for centers in (CENTERS[:3], CENTERS[2:5], CENTERS[[4, 0, 3]]):
        _check_crop(src, top, mask, hm1, centers, cw, ch, fill_value, f"{cw}x{ch} per-sample {centers.tolist()}")
      for one in (CENTERS[3], CENTERS[4:5]):
        _check_crop(src, top, mask, hm1, one, cw, ch, fill_value, f"{cw}x{ch} one centre {one.tolist()}")


@pytest.mark.parametrize("flip", [True, False])
def test_select_offsets_match_single_calls(flip):
  b, C, h, w, cw, ch = 3, 2, 11, 13, 7, 6
  src, top, mask, hm1 = _crop_source(b, C, h, w, 120, None, flip=flip)
  centers = CENTERS[[0, 2, 4]]
  m = src.select(centers, cw, ch)
  assert (m.proj.map_width, m.proj.map_height) == (cw, ch)
  for i in range(b):
    one = dmap.TopdownMap(topdown_map=src.topdown_map[i:i + 1], mask=src.mask[i:i + 1],
                          height_map=src.height_map[i:i + 1],
                          map_projector=src.proj.clone(width_offset=WOFF[i:i + 1].copy(),
                                                       height_offset=HOFF[i:i + 1].copy()))
    s = dmap.crop_topdown_map(one, centers[i:i + 1], cw, ch)
    assert_same(np.asarray(m.proj.width_offset, np.float32).reshape(-1)[i:i + 1],
                np.asarray(s.proj.width_offset, np.float32).reshape(-1), f"width_offset {i}")
    assert_same(np.asarray(m.proj.height_offset, np.float32).reshape(-1)[i:i + 1],
                np.asarray(s.proj.height_offset, np.float32).reshape(-1), f"height_offset {i}")
    assert_same(npy(m.topdown_map[i:i + 1]), npy(s.topdown_map), f"values {i}")


def test_select_multi_pass():
  b, C, h, w = 8, 3, 64, 48
  bound = 3 * pass_items(1)
  side = max(400, math.isqrt(-(-bound // (b * C))) + 1)
  assert b * C * side * side >= bound
  src, top, mask, hm1 = _crop_source(b, C, h, w, 130, -7.0, woff=np.float32(1.0), hoff=np.float32(2.0))
  centers = np.float32([[i * 7.5 - 10, 40 - i * 6.5] for i in range(b)])
  _check_crop(src, top, mask, hm1, centers, side, side, -7.0, f"multi-pass {side}x{side}")


# ---- f. TopdownMap.get_coords / get_points / get_camera / get_origin ----------------------------------------------

@pytest.mark.parametrize("to_global", [True, False])
@pytest.mark.parametrize("flip", [True, False])
def test_topdown_map_coordinates(to_global, flip):
  b, n, Mh, Mw, res = 4, 45, 90, 70, 0.05
  pose = poses(b, 140)
  woff, hoff = WOFF[:b].copy(), HOFF[:b].copy()
  proj = dmap.MapProjector(width=16, height=12, hfov=1.2, cam_pose=pose, width_offset=woff, height_offset=hoff,
                           map_res=res, map_width=Mw, map_height=Mh, to_global=to_global, flip_h=flip)
  m = dmap.TopdownMap(topdown_map=torch.zeros((b, 1, Mh, Mw), device="cuda"),
                      mask=torch.zeros((b, 1, Mh, Mw), dtype=torch.bool, device="cuda"), map_projector=proj)

  def oracle_coords(pts, is_global):
    k = pts.shape[1]
    if to_global and not is_global:
      pts = orc.transform_points(pts, [orc.to_global_steps(pose, k)])
    elif not to_global and is_global:
      pts = orc.transform_points(pts, [orc.from_global_steps(pose, k)])
    return np.stack(orc.map_quantize(pts[..., 0], pts[..., 2], woff, hoff, res, Mh, flip), -1)

  pts = salted((b, n, 3), 141, -3, 3)
  for is_global in (True, False):
    got = twice(lambda: m.get_coords(cu(pts), is_global=is_global))
    assert_same(got, oracle_coords(pts, is_global), f"get_coords is_global={is_global}")
  zero = np.zeros((b, 1, 3), np.float32)
  assert_same(twice(m.get_camera), oracle_coords(zero, False)[:, 0], "get_camera")
  assert_same(twice(m.get_origin), oracle_coords(zero, True)[:, 0], "get_origin")
  coords = np.random.default_rng(142).integers(-100, 200, (b, n, 2))
  got = twice(lambda: m.get_points(cu(coords)))
  x, z = orc.map_dequantize(coords[..., 0], coords[..., 1], woff, hoff, res, Mh, flip)
  assert_same(got, np.stack((x, z), -1), "get_points")


# ---- g. unaligned inputs -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("k", [1, 2, 3])
def test_unaligned_inputs_take_the_scalar_paths(k):
  b, n = 3, 45
  pts = salted((b, n, 3), 150 + k)
  pose = poses(b, 151)
  want = orc.transform_points(pts, [orc.to_global_steps(pose, n)])
  aligned = twice(lambda: dmap.local_to_global_space(cu(pts), pose))
  got = twice(lambda: dmap.local_to_global_space(unaligned(pts, k), pose))
  assert_same(got, want, f"transform at +{k}")
  assert got.tobytes() == aligned.tobytes()
  got = twice(lambda: dmap.utils.rotate(unaligned(pts, k), [0.3, -1.2, 0.5], np.float32([0.4, -1.0, 2.0])))
  assert_same(got, orc.transform_points(pts, [_rot_steps([0.3, -1.2, 0.5], np.float32([0.4, -1.0, 2.0]), n)]),
              f"rotate at +{k}")
  img = _image_points((2, 5, 7, 3), 152)
  for to_image, fn in ((0, dmap.image_to_camera_space), (1, dmap.camera_to_image_space)):
    got = twice(lambda: fn(unaligned(img, k), 23.5, 19.25, 16.0, 12.5))
    assert_same(got, orc.image_camera(img, 23.5, 19.25, 16.0, 12.5, True, 5, to_image), f"{fn.__name__} at +{k}")
    assert got.tobytes() == twice(lambda: fn(cu(img), 23.5, 19.25, 16.0, 12.5)).tobytes()
  shape = (2, 3, 7, 9)
  depth = depth_frames(shape, 153)
  valid = np.random.default_rng(154).random(shape) > 0.3
  got = _check_depth(unaligned(depth, k), valid, unaligned(valid, k), f"depth and valid at +{k}")
  kk = orc.intrinsics(9, 7, math.radians(70))
  ref = twice(lambda: dmap.depth_map_to_point_cloud(cu(depth), cu(valid), kk["fx"], kk["fy"], kk["cx"], kk["cy"],
                                                    TMIN, TMAX, flip_h=False))
  assert got[0].tobytes() == ref[0].tobytes() and got[1].tobytes() == ref[1].tobytes()
