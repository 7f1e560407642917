"""Host-side parameter blocks for the kernels.

The per-sample quantities (poses, pitch, camera height, map offsets) are a few
floats; everything derived from them — the Rodrigues matrices in particular —
is computed here on the CPU with the same torch ops in the same order as the
reference (utils.py:303-327), because sin/cos differ in the last ulp between
CPU and GPU libm and the matrices feed bit-exact bin arithmetic.  The result is
packed as DmStep / DmProjSample / DmFlowSample records (include/dungeon_maps_b200.h)
and uploaded once per distinct parameter set (small LRU cache).
"""
from collections import OrderedDict
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native as nat

ANGLE_EPS = 0.001

STEP_NONE, STEP_ROT_THEN_ADD, STEP_ADD_THEN_ROT, STEP_ADD, STEP_ROT = 0, 1, 2, 3, 4
STEP_WORDS = 16


def host_f32(x, shape_tail=()) -> torch.Tensor:
  """Any scalar / list / ndarray / tensor (any device) → float32 CPU tensor (-1, *shape_tail)."""
  if torch.is_tensor(x):
    t = x.detach()
    if t.dtype is not torch.float32 or t.device.type != "cpu":
      t = t.to(device="cpu", dtype=torch.float32)
  else:
    t = torch.as_tensor(np.asarray(x, dtype=np.float32))
  want = (-1,) + tuple(shape_tail)
  if t.dim() == len(want) and tuple(t.shape[1:]) == want[1:]:
    return t
  return t.reshape(want)


_scalar_rows = {}


def per_sample(x, b: int, shape_tail=(), what: str = "argument") -> torch.Tensor:
  if type(x) is float and shape_tail == ():  # projector defaults repeat call after call
    hit = _scalar_rows.get((x, b))
    if hit is None:
      if len(_scalar_rows) > 256:
        _scalar_rows.clear()
      hit = _scalar_rows[(x, b)] = host_f32(x, ()).expand((b,))
    return hit
  t = host_f32(x, shape_tail)
  if t.shape[0] == b:
    return t
  if t.shape[0] == 1:
    return t.expand((b,) + tuple(shape_tail))
  raise ValueError(f"{what}: expected 1 or {b} entries, got {t.shape[0]}")


def fused_for(n_points: int) -> bool:
  """at::bmm (behind utils.py:329) switches from its naive loop to MKL sgemm at 9*n >= 400;
  the two accumulate differently (see DmStep in the public header)."""
  return 9 * int(n_points) >= 400


_axis_terms = {}


def _skew_terms(axis: Sequence[float]):
  """(skew (1,9), skew² (1,9), I (1,9)) of the normalised axis, utils.py:303-318; they depend on the axis only and
  are built once with the reference's torch ops."""
  key = tuple(float(a) for a in axis)
  hit = _axis_terms.get(key)
  if hit is None:
    ax = host_f32(axis, (3,))
    ax = ax / torch.linalg.norm(ax, dim=-1, keepdim=True)
    zero = torch.zeros((1,), dtype=torch.float32)
    skew = torch.stack((zero, -ax[:, 2], ax[:, 1], ax[:, 2], zero, -ax[:, 0], -ax[:, 1], ax[:, 0], zero), dim=-1)
    skew3 = skew.view(1, 3, 3)
    skew_sq = torch.einsum("bij,bjk->bik", skew3, skew3).reshape(1, 9)
    hit = _axis_terms[key] = (skew.numpy().copy(), skew_sq.numpy().copy(), np.eye(3, dtype=np.float32).reshape(1, 9))
  return hit


def _rotation_matrices_per_sample_axis(ax: torch.Tensor, angle: torch.Tensor, angle_eps: float) -> np.ndarray:
  """utils.rotate with one axis per sample (utils.py:303-327), all in torch like the reference."""
  b = angle.shape[0]
  ax = ax / torch.linalg.norm(ax, dim=-1, keepdim=True)
  if ax.shape[0] != b:
    ax = ax.expand(b, 3)
  zero = torch.zeros((b,), dtype=torch.float32)
  skew = torch.stack((zero, -ax[:, 2], ax[:, 1], ax[:, 2], zero, -ax[:, 0], -ax[:, 1], ax[:, 0], zero), dim=-1)
  skew3 = skew.view(b, 3, 3)
  skew_sq = torch.einsum("bij,bjk->bik", skew3, skew3).reshape(b, 9)
  eye = torch.eye(3, dtype=torch.float32).view(1, 9)
  angle = torch.where(torch.abs(angle) > angle_eps, angle, torch.tensor(0.0))
  return (eye + torch.sin(angle) * skew + (1 - torch.cos(angle)) * skew_sq).numpy()


def rotation_matrices(axis: Sequence[float], angle: torch.Tensor, angle_eps: float = ANGLE_EPS) -> np.ndarray:
  """(b, 9) float32, R = I + sin(a) S + (1 - cos(a)) S², |a| <= eps → identity (utils.py:303-327).
  sin / cos come from torch (the reference's libm path: the last ulp matters); the products and sums around them
  are single IEEE float32 operations in the reference's order, which numpy rounds identically."""
  angle = angle.reshape(-1, 1).to(torch.float32)
  if torch.is_tensor(axis) or isinstance(axis, np.ndarray):
    ax = host_f32(axis, (3,))
    if ax.shape[0] != 1:
      return _rotation_matrices_per_sample_axis(ax, angle, angle_eps)
    axis = ax[0].tolist()
  skew, skew_sq, eye = _skew_terms(axis)
  angle = torch.where(torch.abs(angle) > angle_eps, angle, torch.zeros((), dtype=torch.float32))
  sin, cos = torch.sin(angle).numpy(), torch.cos(angle).numpy()
  return (eye + sin * skew) + (np.float32(1) - cos) * skew_sq


def pack_steps(kind: int, R, t, b: int, n_points: int) -> torch.Tensor:
  """(b, 16) float32 words laid out as DmStep."""
  out = np.zeros((b, STEP_WORDS), dtype=np.float32)
  if kind != STEP_NONE:
    if R is not None:
      out[:, 0:9] = R
    if t is not None:
      out[:, 9:12] = t
    ints = out.view(np.int32)
    ints[:, 12] = kind
    ints[:, 13] = 1 if fused_for(n_points) else 0
  return torch.from_numpy(out)


def xyz(b: int, x=None, y=None, z=None) -> np.ndarray:
  t = np.zeros((b, 3), dtype=np.float32)
  if x is not None: t[:, 0] = np.asarray(x, dtype=np.float32)
  if y is not None: t[:, 1] = np.asarray(y, dtype=np.float32)
  if z is not None: t[:, 2] = np.asarray(z, dtype=np.float32)
  return t


class _StepCache:
  """LRU of packed step blocks keyed by the bytes of their inputs: pitch / camera height repeat call after
  call, poses repeat whenever a caller projects the same frames again.  Entries are read-only."""

  def __init__(self, capacity: int = 256):
    self._d = OrderedDict()
    self._cap = capacity

  def get(self, tag: str, build, n_points: int, *tensors: torch.Tensor) -> torch.Tensor:
    key = (tag, fused_for(n_points)) + tuple(t.contiguous().numpy().tobytes() for t in tensors)
    hit = self._d.get(key)
    if hit is not None:
      self._d.move_to_end(key)
      return hit
    out = build()
    self._d[key] = out
    if len(self._d) > self._cap:
      self._d.popitem(last=False)
    return out


_steps = _StepCache()


def camera_to_local(pitch: torch.Tensor, cam_h: torch.Tensor, n_points: int) -> torch.Tensor:
  b = pitch.shape[0]  # maps.py:789-797
  return _steps.get("c2l", lambda: pack_steps(STEP_ROT_THEN_ADD, rotation_matrices([1., 0., 0.], pitch),
                                              xyz(b, y=cam_h), b, n_points), n_points, pitch, cam_h)


def local_to_camera(pitch: torch.Tensor, cam_h: torch.Tensor, n_points: int) -> torch.Tensor:
  b = pitch.shape[0]  # maps.py:838-845
  return _steps.get("l2c", lambda: pack_steps(STEP_ADD_THEN_ROT, rotation_matrices([1., 0., 0.], -pitch),
                                              xyz(b, y=-cam_h), b, n_points), n_points, pitch, cam_h)


def local_to_global(pose: torch.Tensor, n_points: int) -> torch.Tensor:
  b = pose.shape[0]  # maps.py:883-892
  return _steps.get("l2g", lambda: pack_steps(STEP_ROT_THEN_ADD, rotation_matrices([0., 1., 0.], pose[:, 2]),
                                              xyz(b, x=pose[:, 0], z=pose[:, 1]), b, n_points), n_points, pose)


def global_to_local(pose: torch.Tensor, n_points: int) -> torch.Tensor:
  b = pose.shape[0]  # maps.py:930-939: translate(-pos) then rotate(-yaw)
  return _steps.get("g2l", lambda: pack_steps(STEP_ADD_THEN_ROT, rotation_matrices([0., 1., 0.], -pose[:, 2]),
                                              -xyz(b, x=pose[:, 0], z=pose[:, 1]), b, n_points), n_points, pose)


def identity(b: int) -> torch.Tensor:
  return pack_steps(STEP_NONE, None, None, b, 0)


def fast_steps(samples: torch.Tensor) -> int:
  """DmProjCfg.fast_steps for a (b, 48) block of DmProjSample words: 1 / 2 when every sample's
  steps have the structure the straight-line kernel path assumes (see the public header), else 0."""
  a = samples.numpy()
  ints = a.view(np.int32)
  local_ok = ((ints[:, 12:14] == (STEP_ROT_THEN_ADD, 1)).all() and (a[:, 0] == 1).all()
              and not a[:, (1, 2, 3, 6, 9, 11)].any())
  if not local_ok:
    return 0
  if not ints[:, 28].any():  # STEP_NONE
    return 1
  global_ok = ((ints[:, 28:30] == (STEP_ROT_THEN_ADD, 1)).all() and (a[:, 16 + 4] == 1).all()
               and not a[:, (16 + 1, 16 + 3, 16 + 5, 16 + 7, 16 + 10)].any())
  return 2 if global_ok else 0


# ---- the same blocks packed in C (csrc/dm_params.cu) ------------------------------------------------------------
# For the common case — one cam_pitch / cam_height for the whole batch — the per-sample blocks are a function of the
# poses alone, and building them with torch / numpy cost 0.1-0.25 ms of interpreter time per call.  The C packers form
# the yaw rotation from torch's own sin / cos (computed here) with the reference's float32 operation order.

_pose_cfgs = {}


def _uniform(t: torch.Tensor) -> bool:
  """All entries of a per-sample tensor are one value (a scalar that per_sample expanded, or b == 1)."""
  return t.dim() == 1 and (t.shape[0] == 1 or t.stride(0) == 0)


def pose_cfg(pitch: torch.Tensor, cam_h: torch.Tensor, n_points: int) -> "nat.DmPoseCfg":
  key = (float(pitch[0]), float(cam_h[0]), fused_for(n_points))
  cfg = _pose_cfgs.get(key)
  if cfg is None:
    cfg = nat.DmPoseCfg()
    p1 = pitch[:1].contiguous()
    cfg.pitch_R[:] = rotation_matrices([1., 0., 0.], p1).reshape(-1).tolist()        # maps.py:789-793
    cfg.pitch_back_R[:] = rotation_matrices([1., 0., 0.], -p1).reshape(-1).tolist()  # maps.py:838-842
    cfg.cam_height = float(cam_h[0])
    skew, skew_sq, _ = _skew_terms([0., 1., 0.])
    cfg.yaw_skew[:] = skew.reshape(-1).tolist()
    cfg.yaw_skew_sq[:] = skew_sq.reshape(-1).tolist()
    cfg.fused = int(fused_for(n_points))
    if len(_pose_cfgs) > 64:
      _pose_cfgs.clear()
    _pose_cfgs[key] = cfg
  return cfg


def yaw_sin_cos(pose: torch.Tensor):
  """sin / cos of the yaw column with the reference's torch-CPU ops (utils.py:325-326); contiguous float32 CPU tensors.
  The |a| <= ANGLE_EPS → 0 clamp (utils.py:323-324) is applied by the C packers, which replace the pair by exactly
  (0, 1) = (sin 0, cos 0) for such angles."""
  yaw = pose[:, 2]
  return torch.sin(yaw), torch.cos(yaw)


def proj_samples(pose, pitch, cam_h, woff, hoff, to_global: bool, n_points: int):
  """(b, 48) float32 DmProjSample words + DmProjCfg.fast_steps for orth_project."""
  b = pose.shape[0]
  if _uniform(pitch) and _uniform(cam_h):
    out = torch.empty((b, nat.PROJ_SAMPLE_WORDS), dtype=torch.float32)
    fast = nat.c_int32(0)
    woff, hoff = woff.contiguous(), hoff.contiguous()
    if to_global:
      pose = pose.contiguous()
      sin, cos = yaw_sin_cos(pose)
      rc = nat.lib().dm_pack_proj_samples(pose_cfg(pitch, cam_h, n_points), pose.data_ptr(), sin.data_ptr(),
                                          cos.data_ptr(), woff.data_ptr(), hoff.data_ptr(), 1, b, out.data_ptr(),
                                          nat.ctypes.byref(fast))
    else:
      rc = nat.lib().dm_pack_proj_samples(pose_cfg(pitch, cam_h, n_points), None, None, None, woff.data_ptr(),
                                          hoff.data_ptr(), 0, b, out.data_ptr(), nat.ctypes.byref(fast))
    nat.check(rc, "dm_pack_proj_samples")
    return out, fast.value
  samples = torch.zeros((b, nat.PROJ_SAMPLE_WORDS), dtype=torch.float32)
  samples[:, 0:16] = camera_to_local(pitch, cam_h, n_points)
  samples[:, 16:32] = local_to_global(pose, n_points) if to_global else identity(b)
  samples[:, 32] = woff
  samples[:, 33] = hoff
  return samples, fast_steps(samples)


def flow_samples(pose, pitch, cam_h, n_points: int) -> torch.Tensor:
  """(b, 48) float32 DmFlowSample words for camera_affine_grid."""
  b = pose.shape[0]
  if _uniform(pitch) and _uniform(cam_h):
    out = torch.empty((b, nat.FLOW_SAMPLE_WORDS), dtype=torch.float32)
    pose = pose.contiguous()
    sin, cos = yaw_sin_cos(pose)
    nat.check(nat.lib().dm_pack_flow_samples(pose_cfg(pitch, cam_h, n_points), pose.data_ptr(), sin.data_ptr(),
                                             cos.data_ptr(), b, out.data_ptr()), "dm_pack_flow_samples")
    return out
  return torch.cat((camera_to_local(pitch, cam_h, n_points), local_to_global(pose, n_points),
                    local_to_camera(pitch, cam_h, n_points)), dim=1)


_ego_cfgs = {}


def ego_samples(pose, src_woff, src_hoff, woff, hoff, n_points: int) -> torch.Tensor:
  """(b, 20) float32 words of TopdownMap.select_egocentric (DM_EGO_SAMPLE_WORDS): local_to_global(pose, n_points) as a
  DmStep, then the source map's offsets, then the window's.  Packed in C from torch's sin / cos of the yaws."""
  fused = int(fused_for(n_points))
  cfg = _ego_cfgs.get(fused)
  if cfg is None:  # the packer reads the yaw terms and `fused` only
    cfg = nat.DmPoseCfg()
    skew, skew_sq, _ = _skew_terms([0., 1., 0.])
    cfg.yaw_skew[:] = skew.reshape(-1).tolist()
    cfg.yaw_skew_sq[:] = skew_sq.reshape(-1).tolist()
    cfg.fused = fused
    _ego_cfgs[fused] = cfg
  b = pose.shape[0]
  pose = pose.contiguous()
  sin, cos = yaw_sin_cos(pose)
  cols = [t.contiguous() for t in (src_woff, src_hoff, woff, hoff)]
  out = torch.empty((b, nat.EGO_SAMPLE_WORDS), dtype=torch.float32)
  nat.check(nat.lib().dm_pack_ego_samples(cfg, pose.data_ptr(), sin.data_ptr(), cos.data_ptr(),
                                          *[t.data_ptr() for t in cols], b, out.data_ptr()), "dm_pack_ego_samples")
  return out


class DeviceBlock:
  """A parameter block uploaded by dm_upload_params: a raw device pointer into the library's ring of slots, valid for
  the work queued on the current stream before the 64th upload after it (every caller hands it to the very next C
  call).  Quacks like the tensor the callers used to get: data_ptr()."""
  __slots__ = ("ptr", "nbytes")

  def __init__(self, ptr: int, nbytes: int):
    self.ptr, self.nbytes = ptr, nbytes

  def data_ptr(self) -> int:
    return self.ptr


_UPLOAD_MAX = 64 * 1024  # kUpSlotBytes of csrc/dm_api.cu


def upload(host: torch.Tensor, device: torch.device):
  """Device copy of a host parameter block for the next call queued on the current stream: the library's pinned ring
  and copy stream (dm_upload_params; a torch copy on the caller's stream put a copy-engine round trip between the
  kernels of consecutive calls and cost ~50 us of host time).  Blocks above 64 KiB (thousands of samples) go through
  torch.  Returns an object with data_ptr()."""
  host = host.contiguous()
  nbytes = host.numel() * host.element_size()
  if nbytes == 0 or nbytes > _UPLOAD_MAX:
    return host.to(device)
  out = nat.c_void_p()
  with torch.cuda.device(device):
    rc = nat.lib().dm_upload_params(host.data_ptr(), nbytes, nat.stream_ptr(device), nat.ctypes.byref(out))
  nat.check(rc, "dm_upload_params")
  return DeviceBlock(out.value, nbytes)
