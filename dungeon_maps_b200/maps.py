"""Drop-in for `dungeon_maps.maps` (reference: /root/reference/dungeon_maps/maps.py).

Same public functions and classes, same argument names / meaning / defaults;
the bodies call the fused sm_100a kernels through the C ABI
(include/dungeon_maps_b200.h) instead of chaining ~100 aten ops and
torch_scatter.  Host code here only validates and reshapes arguments, builds
the per-sample parameter blocks (_params.py) and allocates outputs.

There is no CPU path: inputs that are not on a CUDA device are moved to one
(`device=` or the current CUDA device); results live on that device.  Batch > 1
is supported and defined as "the reference applied to every sample"
(the reference itself raises for batch > 1, utils.py:311-316).
"""
import copy
import enum
import inspect
from typing import Any, Dict, List, Optional, Tuple, Union

import numpy as np
import torch

from . import _native as nat
from . import _params as prm
from . import utils
from .utils import CameraIntrinsics, Float3D, NINF, Reduction


@enum.unique
class CenterMode(str, enum.Enum):
  """maps.py:26-39; CenterMode(None) is CenterMode.none."""
  none = "none"
  origin = "origin"
  camera = "camera"

  @classmethod
  def _missing_(cls, value):
    if value is None:
      return cls.none


__all__ = [
  'CenterMode', 'get', 'orth_project', 'camera_affine_grid', 'compute_ego_flow', 'depth_map_to_point_cloud',
  'height_map_to_point_cloud', 'image_to_camera_space', 'camera_to_image_space', 'camera_to_local_space',
  'local_to_camera_space', 'local_to_global_space', 'global_to_local_space', 'map_quantize',
  'map_dequantize', 'project', 'compute_center_offsets', 'MapProjector', 'TopdownMap', 'crop_topdown_map',
  'crop_egocentric_map', 'score_poses', 'geodesic_distance', 'connected_components', 'distance_transform', 'fuse_topdown_maps',
  'merge_into_canvas', 'MapBuilder', 'release_workspaces', 'Reduction', 'CameraIntrinsics', 'NINF', 'Float3D',
]


def get(*args: Any) -> Any:
  """First argument that is not None (the last one if all are)."""
  arg = None
  for arg in args:
    if arg is not None:
      break
  return arg


# ---- internal plumbing ----------------------------------------------------------------------

_workspaces: Dict[Tuple[int, int], torch.Tensor] = {}


def _workspace(dev: torch.device, nbytes: int) -> torch.Tensor:
  """Zero-initialised accumulation ring, one per (device, stream); the kernels leave it zeroed."""
  key = (dev.index, nat.stream_ptr(dev))
  ws = _workspaces.get(key)
  if ws is None or ws.numel() < nbytes:
    ws = torch.zeros(max(nbytes, 16), dtype=torch.uint8, device=dev)
    _workspaces[key] = ws
  return ws


def _alloc_canvas(shape: Tuple[int, ...], dtype: torch.dtype, dev: torch.device) -> torch.Tensor:
  """A fresh, contiguous tensor of `shape` for a map whose size is data dependent (the merged world map grows step by
  step, maps.py:2171-2178).  The storage is rounded up to a size class (a quarter of a power of two apart): torch's
  caching allocator can then hand the block a merge freed two steps ago to the next, slightly larger map instead of
  going to cudaMalloc — a device-wide synchronising call, twice per step — for every new size."""
  n = int(np.prod(shape))
  if n < (1 << 18):
    return torch.empty(shape, dtype=dtype, device=dev)
  return torch.empty((_canvas_cap(n),), dtype=dtype, device=dev)[:n].view(shape)


def _canvas_cap(n: int) -> int:
  """Size class of a canvas of n elements: the next of {5/8, 6/8, 7/8, 8/8} of the power of two above n."""
  top = 1 << (n - 1).bit_length()          # smallest power of two >= n
  return next(c for c in (top // 2 + k * (top // 8) for k in range(1, 5)) if c >= n)


def release_workspaces() -> None:
  """Frees the cached accumulation rings (one per device and stream that projected something) and the library's
  own scratch of the host-buffer entries."""
  _workspaces.clear()
  nat.lib().dm_release_scratch()


def _pick_device(device, *tensors) -> torch.device:
  if device is not None and not isinstance(device, bool):
    return nat.require_cuda(device)
  for t in tensors:
    if torch.is_tensor(t) and t.is_cuda:
      return t.device
  return nat.require_cuda(None)


def _image(x, dev: torch.device, dtype: torch.dtype) -> torch.Tensor:
  """2/3/4-D image → contiguous (b, c, h, w) on `dev`."""
  t = utils.to_tensor(x)
  t = utils.to_4D_image(t)
  return t.to(device=dev, dtype=dtype).contiguous()


def _points(x, dev: torch.device) -> Tuple[torch.Tensor, torch.Size]:
  """(..., 3) points → contiguous (b, n, 3) float32 on `dev` plus the original shape."""
  t = utils.to_tensor(x).to(device=dev, dtype=torch.float32)
  shape = t.shape
  if t.dim() < 2:
    t = t.view(-1, 3)
  b = t.shape[0]
  return t.reshape(b, -1, 3).contiguous(), shape


def _run_steps(points, dev, host_steps: List[torch.Tensor]) -> torch.Tensor:
  flat, shape = _points(points, dev)
  steps = torch.cat(host_steps, dim=1)
  return utils._apply_steps(flat, steps, len(host_steps)).reshape(shape)


def _f32(x) -> float:
  """Python float rounded to float32 (what torch does to a Python scalar in a float32 op)."""
  return float(np.float32(x))


# ======== Raw functional APIs (maps.py:121-1248) ==============================================

def orth_project(
  depth_map: torch.Tensor,
  value_map: Optional[torch.Tensor],
  valid_map: Optional[torch.Tensor],
  cam_pose: torch.Tensor,
  width_offset: torch.Tensor,
  height_offset: torch.Tensor,
  cam_pitch: torch.Tensor,
  cam_height: torch.Tensor,
  map_res: float,
  map_width: int,
  map_height: int,
  focal_x: float,
  focal_y: float,
  center_x: float,
  center_y: float,
  trunc_depth_min: Optional[float],
  trunc_depth_max: Optional[float],
  trunc_height_max: Optional[float],
  clip_border: Optional[int],
  to_global: bool,
  flip_h: bool = True,
  fill_value: Optional[float] = None,
  reduction: Optional[Reduction] = None,
  get_height_map: bool = False,
  device: Optional[torch.device] = None,
  _validate_args: bool = True,
  label_map: Optional[torch.Tensor] = None,
  num_classes: Optional[int] = None
) -> Union[Tuple[torch.Tensor, torch.Tensor], Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]:
  """Orthographic projection of UNNORMALIZED depth maps (and optional per-pixel value maps)
  onto top-down maps: one fused kernel pass + one resolve pass (csrc/dm_project.cu) in place of
  maps.py:259-351.  Arguments, defaults and return values are those of the reference:

  Returns (topdown_map (b,C,mh,mw) f32, masks (b,C,mh,mw) bool[, height_map]); every value
  channel is reduced independently (max unless `reduction` says min); cells nothing landed on
  hold `fill_value` (0 when None) and are False in `masks`; `height_map` is the same tensor as
  `topdown_map` when `value_map` is None, otherwise a stride-0 expand of the (b,1,mh,mw)
  max-height map with -inf in empty cells.

  Addition to the reference's signature: `label_map` (b, 1, h, w) integer class ids with `num_classes` = C gives,
  bit for bit, the result of value_map = one_hot(label_map, C) as float32 planes (what the reference's object-map
  demo builds, demos/object_map/run.py:117-124) without ever materialising those planes — csrc/dm_labels.cu.
  """
  if label_map is not None:
    if value_map is not None:
      raise ValueError("pass either `value_map` or `label_map`, not both")
    if num_classes is None:
      raise ValueError("`label_map` needs `num_classes` (the C of one_hot(label_map, C))")
    if not 1 <= int(num_classes) <= 63:
      raise ValueError(f"num_classes must be in 1..63, got {num_classes}")
  if utils._reduction_code(reduction, fused=False) > 1:
    if label_map is not None:  # rarely used reductions: materialise the one-hot planes and take the composed path
      value_map = _one_hot_planes(label_map, int(num_classes), _pick_device(device, depth_map, label_map))
    return _orth_project_composed(
      depth_map, value_map, valid_map, cam_pose, width_offset, height_offset, cam_pitch, cam_height, map_res,
      map_width, map_height, focal_x, focal_y, center_x, center_y, trunc_depth_min, trunc_depth_max,
      trunc_height_max, clip_border, to_global, flip_h, fill_value, reduction, get_height_map, device)
  red = utils._reduction_code(reduction)
  dev = _pick_device(device, depth_map, value_map, label_map)
  depth = _image(depth_map, dev, torch.float32)
  b, dc, H, W = depth.shape
  values = None if value_map is None else _batch_of(_image(value_map, dev, torch.float32), b, "value_map")
  valid = None if valid_map is None else _batch_of(_image(valid_map, dev, torch.bool), b, "valid_map")
  labels = None if label_map is None else _batch_of(_label_ids(label_map, int(num_classes), dev), b, "label_map")
  for name, t in (("value_map", values), ("valid_map", valid), ("label_map", labels)):
    if t is not None and t.shape[-2:] != depth.shape[-2:]:
      raise RuntimeError(f"{name} {tuple(t.shape)} does not match depth_map {tuple(depth.shape)}")
  if labels is not None and (dc != 1 or labels.shape[1] != 1):
    raise RuntimeError("label_map needs single-channel depth and label maps: (b, 1, h, w)")
  # per-sample host parameters
  pose = prm.per_sample(cam_pose, b, (3,), "cam_pose")
  pitch = prm.per_sample(cam_pitch, b, (), "cam_pitch")
  camh = prm.per_sample(cam_height, b, (), "cam_height")
  woff = prm.per_sample(width_offset, b, (), "width_offset")
  hoff = prm.per_sample(height_offset, b, (), "height_offset")
  frames = b
  C = int(num_classes) if labels is not None else (0 if values is None else values.shape[1])
  if dc != 1:
    # one index set per depth channel (maps.py:298-318 keeps the channel dim): fold it into the batch
    if values is not None and values.shape[1] != dc:
      raise RuntimeError(f"value_map has {values.shape[1]} channels, depth_map has {dc}")
    if valid is not None and valid.shape[1] not in (1, dc):
      raise RuntimeError(f"valid_map has {valid.shape[1]} channels, depth_map has {dc}")
    frames = b * dc
    depth = depth.reshape(frames, 1, H, W)
    if values is not None:
      values = values.reshape(frames, 1, H, W)
      C = 1
    if valid is not None:
      valid = valid.expand(b, dc, H, W).reshape(frames, 1, H, W).contiguous()
    rep = lambda t: t.repeat_interleave(dc, dim=0)
    pose, pitch, camh, woff, hoff = rep(pose), rep(pitch), rep(camh), rep(woff), rep(hoff)
  elif valid is not None and valid.shape[1] != 1:
    raise RuntimeError(f"valid_map has {valid.shape[1]} channels, depth_map has 1")
  n_points = dc * H * W  # points the reference rotates per sample in one bmm
  samples, fast_steps = prm.proj_samples(pose, pitch, camh, woff, hoff, bool(to_global), n_points)
  samples_dev = prm.upload(samples, dev)

  cfg = nat.DmProjCfg()
  cfg.H, cfg.W, cfg.C, cfg.Mh, cfg.Mw = H, W, C, int(map_height), int(map_width)
  cfg.fx, cfg.fy, cfg.cx, cfg.cy = focal_x, focal_y, center_x, center_y
  cfg.map_res = map_res
  cfg.has_trunc_depth_min = trunc_depth_min is not None
  cfg.has_trunc_depth_max = trunc_depth_max is not None
  cfg.has_trunc_height_max = trunc_height_max is not None
  cfg.trunc_depth_min = trunc_depth_min or 0.
  cfg.trunc_depth_max = trunc_depth_max or 0.
  cfg.trunc_height_max = trunc_height_max or 0.
  cfg.clip_border = int(clip_border) if clip_border is not None else 0
  cfg.flip_h = bool(flip_h)
  cfg.fill_value = 0. if fill_value is None else fill_value
  want_height = bool(get_height_map) and C > 0
  cfg.want_height = want_height
  cfg.reduction = red
  cfg.fast_steps = fast_steps
  Cv = max(C, 1)
  topdown = torch.empty((frames, Cv, cfg.Mh, cfg.Mw), dtype=torch.float32, device=dev)
  masks = torch.empty((frames, Cv, cfg.Mh, cfg.Mw), dtype=torch.bool, device=dev)
  height = torch.empty((frames, 1, cfg.Mh, cfg.Mw), dtype=torch.float32, device=dev) if want_height else None
  lib = nat.lib()
  with torch.cuda.device(dev):
    if labels is not None:
      ws = _workspace(dev, lib.dm_orth_project_labels_workspace_bytes(cfg, frames))
      rc = lib.dm_orth_project_labels_f32(depth.data_ptr(), labels.data_ptr(), nat.ptr(valid), samples_dev.data_ptr(),
                                          cfg, frames, topdown.data_ptr(), masks.data_ptr(), nat.ptr(height),
                                          ws.data_ptr(), ws.numel(), nat.stream_ptr(dev))
      nat.check(rc, "dm_orth_project_labels_f32")
    else:
      ws = _workspace(dev, lib.dm_orth_project_workspace_bytes(cfg, frames))
      rc = lib.dm_orth_project_f32(depth.data_ptr(), nat.ptr(values), nat.ptr(valid), samples_dev.data_ptr(),
                                   cfg, frames, topdown.data_ptr(), masks.data_ptr(), nat.ptr(height),
                                   ws.data_ptr(), ws.numel(), nat.stream_ptr(dev))
      nat.check(rc, "dm_orth_project_f32")
  if dc != 1:
    topdown = topdown.reshape(b, dc, cfg.Mh, cfg.Mw)
    masks = masks.reshape(b, dc, cfg.Mh, cfg.Mw)
    if height is not None:
      height = height.reshape(b, dc, cfg.Mh, cfg.Mw)
  if not get_height_map:
    return topdown, masks
  if C == 0:
    return topdown, masks, topdown          # maps.py:333-334: the very same tensor
  return topdown, masks, torch.broadcast_to(height, topdown.shape)  # maps.py:349


def _batch_of(t: torch.Tensor, b: int, what: str) -> torch.Tensor:
  """A per-frame image tensor with batch 1 is shared by all b frames (the reference's ops broadcast it); the kernels
  index every plane by frame, so it is expanded here."""
  if t.shape[0] == b:
    return t
  if t.shape[0] == 1:
    return t.expand((b,) + tuple(t.shape[1:])).contiguous()
  raise RuntimeError(f"{what} has batch {t.shape[0]}, depth_map has batch {b}")


def _label_ids(label_map, num_classes: int, dev: torch.device) -> torch.Tensor:
  """Class ids as the kernels take them: contiguous (b, 1, h, w) uint8 on `dev`; ids outside [0, num_classes)
  become 255 ("no class": an all-zero one-hot row).  uint8 input is used as it is."""
  t = utils.to_4D_image(utils.to_tensor(label_map))
  if t.dtype is not torch.uint8:
    if t.dtype.is_floating_point or t.dtype is torch.bool:
      raise TypeError(f"label_map must hold integer class ids, got {t.dtype}")
    t = t.to(dev)
    t = torch.where((t < 0) | (t >= num_classes), torch.full_like(t, 255), t).to(torch.uint8)
  return t.to(dev).contiguous()


def _one_hot_planes(label_map, num_classes: int, dev: torch.device) -> torch.Tensor:
  ids = _label_ids(label_map, num_classes, dev)[:, 0].to(torch.int64)               # (b, h, w)
  planes = torch.arange(num_classes, device=dev).view(1, -1, 1, 1) == ids.unsqueeze(1)
  return planes.to(torch.float32)


def _orth_project_composed(depth_map, value_map, valid_map, cam_pose, width_offset, height_offset, cam_pitch,
                            cam_height, map_res, map_width, map_height, focal_x, focal_y, center_x, center_y,
                            trunc_depth_min, trunc_depth_max, trunc_height_max, clip_border, to_global, flip_h,
                            fill_value, reduction, get_height_map, device):
  """orth_project for the reductions the fused kernel does not cover (sum, mean, prod): the reference's own
  sequence of public steps (maps.py:259-351), each of them one kernel of this package — points are materialised
  here, the price of the rarely used reductions."""
  dev = _pick_device(device, depth_map, value_map)
  depth = _image(depth_map, dev, torch.float32)
  b, dc, H, W = depth.shape
  points, valid = depth_map_to_point_cloud(depth, valid_map, focal_x, focal_y, center_x, center_y, trunc_depth_min,
                                           trunc_depth_max, flip_h, device=dev)          # (b, c, h, w, 3)
  if clip_border is not None and clip_border > 0:                                        # maps.py:48-70
    k = int(clip_border)
    border = torch.zeros((H, W), dtype=torch.bool, device=dev)
    border[k:H - k, k:W - k] = True
    valid = valid & border
  points = camera_to_local_space(points, cam_pitch, cam_height, device=dev)
  if trunc_height_max is not None:                                                       # maps.py:286-288
    valid = valid & (points[..., 1] <= trunc_height_max)
  if to_global:
    points = local_to_global_space(points, cam_pose, device=dev)
  flat = points.reshape(b, dc, H * W, 3)
  flat_mask = valid.reshape(b, dc, H * W)
  x_bin, z_bin = map_quantize(flat[..., 0].reshape(b, -1), flat[..., 2].reshape(b, -1), width_offset, height_offset,
                              map_res, map_height, flip_h, device=dev)
  coords = torch.stack((z_bin, x_bin), dim=-1).reshape(b, dc, H * W, 2)
  heights = flat[..., 1]
  values = heights if value_map is None else _image(value_map, dev, torch.float32).reshape(b, -1, H * W)
  canvas = torch.zeros(values.shape[:-1] + (int(map_height), int(map_width)), dtype=torch.float32, device=dev)
  topdown, masks = project(coords, values, flat_mask, canvas, fill_value=fill_value, reduction=reduction, device=dev)
  if not get_height_map:
    return topdown, masks
  if value_map is None:
    return topdown, masks, topdown                                                       # maps.py:333-334
  hcanvas = torch.zeros((b, dc, int(map_height), int(map_width)), dtype=torch.float32, device=dev)
  height, _ = project(coords, heights, flat_mask, hcanvas, fill_value=NINF, reduction=Reduction.max, device=dev)
  return topdown, masks, torch.broadcast_to(height, topdown.shape)                       # maps.py:349


def camera_affine_grid(
  depth_map: torch.Tensor,
  trans_pose: torch.Tensor,
  cam_pitch: torch.Tensor,
  cam_height: torch.Tensor,
  focal_x: float,
  focal_y: float,
  center_x: float,
  center_y: float,
  flip_h: bool = True,
  device: Optional[torch.device] = None,
  _validate_args: bool = True,
  _emit_flow: bool = False
) -> torch.Tensor:
  """Where every pixel of `depth_map` (time t) lands in the image after the camera moved by
  `trans_pose` = [dx, dz, dyaw]: one fused element-wise kernel (csrc/dm_flow.cu) in place of
  maps.py:414-460.  Returns the (b, ..., h, w, 2) float32 grid of image (x, y)."""
  dev = _pick_device(device, depth_map)
  depth = _image(depth_map, dev, torch.float32)
  b, ch, H, W = depth.shape
  pose = prm.per_sample(trans_pose, b, (3,), "trans_pose")
  pitch = prm.per_sample(cam_pitch, b, (), "cam_pitch")
  camh = prm.per_sample(cam_height, b, (), "cam_height")
  n_points = ch * H * W
  samples_dev = prm.upload(prm.flow_samples(pose, pitch, camh, n_points), dev)
  cfg = nat.DmFlowCfg()
  cfg.H, cfg.W, cfg.channels = H, W, ch
  cfg.fx, cfg.fy, cfg.cx, cfg.cy = focal_x, focal_y, center_x, center_y
  cfg.flip_h = bool(flip_h)
  cfg.emit_flow = bool(_emit_flow)
  grid = torch.empty((b, ch, H, W, 2), dtype=torch.float32, device=dev)
  with torch.cuda.device(dev):
    rc = nat.lib().dm_affine_grid_f32(depth.data_ptr(), samples_dev.data_ptr(), cfg, b, grid.data_ptr(),
                                      nat.stream_ptr(dev))
  nat.check(rc, "dm_affine_grid_f32")
  return grid


def compute_ego_flow(proj: "MapProjector", depth_map: torch.Tensor, trans_pose: torch.Tensor) -> torch.Tensor:
  """Egocentric motion flow of the reference's demo helper (demos/ego_flow/run.py:75-90):
  (x - grid_x, -(y - grid_y)) in pixels, fused into the same kernel.  depth_map (c, h, w) or
  (b, c, h, w); returns the flow of the first sample / channel, (h, w, 2), like the demo."""
  flow = camera_affine_grid(
    depth_map=depth_map, trans_pose=trans_pose, cam_pitch=proj.cam_pitch, cam_height=proj.cam_height,
    focal_x=proj.cam_params.fx, focal_y=proj.cam_params.fy, center_x=proj.cam_params.cx,
    center_y=proj.cam_params.cy, flip_h=proj.flip_h, device=proj.device, _emit_flow=True)
  return flow[0, 0]


def depth_map_to_point_cloud(
  depth_map: torch.Tensor,
  valid_map: Optional[torch.Tensor],
  focal_x: float,
  focal_y: float,
  center_x: float,
  center_y: float,
  trunc_depth_min: Optional[float],
  trunc_depth_max: Optional[float],
  flip_h: bool = True,
  device: Optional[torch.device] = None,
  _validate_args: bool = True
) -> Tuple[torch.Tensor, torch.Tensor]:
  """Camera-space points (b, c, h, w, 3) and the valid area (b, c, h, w) of a depth map
  (maps.py:462-545); X right, Y up, Z forward."""
  dev = _pick_device(device, depth_map)
  depth = _image(depth_map, dev, torch.float32)
  b, c, H, W = depth.shape
  valid = None
  if valid_map is not None:
    valid = _image(valid_map, dev, torch.bool).expand(b, c, H, W).contiguous()
  pts = torch.empty((b, c, H, W, 3), dtype=torch.float32, device=dev)
  ok = torch.empty((b, c, H, W), dtype=torch.bool, device=dev)
  with torch.cuda.device(dev):
    rc = nat.lib().dm_depth_to_points_f32(
      depth.data_ptr(), nat.ptr(valid), b * c, H, W, focal_x, focal_y, center_x, center_y, int(bool(flip_h)),
      int(trunc_depth_min is not None), trunc_depth_min or 0., int(trunc_depth_max is not None),
      trunc_depth_max or 0., pts.data_ptr(), ok.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_depth_to_points_f32")
  return pts, ok


def height_map_to_point_cloud(
  height_map: torch.Tensor,
  width_offset: torch.Tensor,
  height_offset: torch.Tensor,
  map_res: float,
  map_height: int,
  flip_h: bool = True,
  device: Optional[torch.device] = None,
  _validate_args: bool = True
) -> torch.Tensor:
  """Every cell of a height map as a 3-D point (b, c, h, w, 3) (maps.py:547-612)."""
  dev = _pick_device(device, height_map)
  hm = _image(height_map, dev, torch.float32)
  xb, zb = utils.generate_image_coords(hm.shape, dtype=torch.float32, device=dev)
  x, z = map_dequantize(xb, zb, width_offset, height_offset, map_res, map_height, flip_h, device=dev)
  return torch.stack((x, hm, z), dim=-1)


def _image_camera(points, fx, fy, cx, cy, flip_h, height, to_image, device):
  dev = _pick_device(device, points)
  t = utils.to_tensor(points).to(device=dev, dtype=torch.float32)
  if flip_h and height is None:
    if t.dim() < 3:
      raise RuntimeError("The rank of `points` must be at least 3D (..., h, w, 3) "
                         "or `height` should be provided if `flip_h` is enabled.")
    height = t.shape[-3]
  flat = t.reshape(-1, 3).contiguous()
  out = torch.empty_like(flat)
  with torch.cuda.device(dev):
    rc = nat.lib().dm_image_camera_f32(flat.data_ptr(), flat.shape[0], fx, fy, cx, cy, int(bool(flip_h)),
                                       int(height or 0), int(to_image), out.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_image_camera_f32")
  return out.reshape(t.shape)


def image_to_camera_space(points: torch.Tensor, focal_x: float, focal_y: float, center_x: float,
                          center_y: float, flip_h: bool = True, height: Optional[int] = None,
                          device: Optional[torch.device] = None, _validate_args: bool = True) -> torch.Tensor:
  """(pixel x, pixel y, depth) → camera space (maps.py:616-682)."""
  return _image_camera(points, focal_x, focal_y, center_x, center_y, flip_h, height, 0, device)


def camera_to_image_space(points: torch.Tensor, focal_x: float, focal_y: float, center_x: float,
                          center_y: float, flip_h: bool = True, height: Optional[int] = None,
                          device: Optional[torch.device] = None, _validate_args: bool = True) -> torch.Tensor:
  """Camera space → (pixel x, pixel y, depth) (maps.py:684-751)."""
  return _image_camera(points, focal_x, focal_y, center_x, center_y, flip_h, height, 1, device)


def _n_points(points) -> Tuple[int, int]:
  t = utils.to_tensor(points)
  if t.dim() < 2:
    return 1, max(t.numel() // 3, 1)
  b = t.shape[0]
  return b, max(t.numel() // (3 * max(b, 1)), 1)


def _per_sample_steps(points, build, *params):
  """Step blocks for a transform whose per-sample parameters (pose, pitch, height) may carry a batch of their own:
  like the reference's tensor ops, a single point set is broadcast over b parameter sets (TopdownMap.get_camera of
  a batched map, maps.py:1824-1839) and a single parameter set over b point sets.  Returns (points, steps)."""
  bp, n = _n_points(points)
  tails = [(3,) if isinstance(p, tuple) else () for p in params]
  vals = [prm.host_f32(p[0] if isinstance(p, tuple) else p, tail) for p, tail in zip(params, tails)]
  b = max([bp] + [v.shape[0] for v in vals])
  if bp != b:
    t = utils.to_tensor(points)
    if bp != 1:
      raise ValueError(f"points have batch {bp}, the transform parameters {b}")
    if t.dim() < 2:
      t = t.view(1, -1, 3)
    points = t.expand((b,) + tuple(t.shape[1:]))
  args = [prm.per_sample(v, b, tail) for v, tail in zip(vals, tails)]
  return points, build(*args, n)


def camera_to_local_space(points: torch.Tensor, cam_pitch: torch.Tensor, cam_height: torch.Tensor,
                          device: Optional[torch.device] = None, _validate_args: bool = True) -> torch.Tensor:
  """Rotate by the camera pitch about x, lift by the camera height (maps.py:753-800)."""
  points, st = _per_sample_steps(points, prm.camera_to_local, cam_pitch, cam_height)
  return _run_steps(points, _pick_device(device, points), [st])


def local_to_camera_space(points: torch.Tensor, cam_pitch: torch.Tensor, cam_height: torch.Tensor,
                          device: Optional[torch.device] = None, _validate_args: bool = True) -> torch.Tensor:
  """Inverse of camera_to_local_space (maps.py:802-848)."""
  points, st = _per_sample_steps(points, prm.local_to_camera, cam_pitch, cam_height)
  return _run_steps(points, _pick_device(device, points), [st])


def local_to_global_space(points: torch.Tensor, cam_pose: torch.Tensor,
                          device: Optional[torch.device] = None, _validate_args: bool = True) -> torch.Tensor:
  """Rotate by yaw about y, translate by (x, 0, z) (maps.py:850-895)."""
  points, st = _per_sample_steps(points, prm.local_to_global, (cam_pose,))
  return _run_steps(points, _pick_device(device, points), [st])


def global_to_local_space(points: torch.Tensor, cam_pose: torch.Tensor,
                          device: Optional[torch.device] = None, _validate_args: bool = True) -> torch.Tensor:
  """Inverse of local_to_global_space (maps.py:897-942)."""
  points, st = _per_sample_steps(points, prm.global_to_local, (cam_pose,))
  return _run_steps(points, _pick_device(device, points), [st])


def _coords_pair(x_coords, z_coords, dev):
  x = utils.to_tensor(x_coords).to(device=dev, dtype=torch.float32)
  z = utils.to_tensor(z_coords).to(device=dev, dtype=torch.float32)
  x, z = torch.broadcast_tensors(x, z)
  shape = x.shape
  if x.dim() < 2:
    x, z = x.reshape(1, -1), z.reshape(1, -1)
  b = x.shape[0]
  return x.reshape(b, -1).contiguous(), z.reshape(b, -1).contiguous(), shape, b


def map_quantize(x_coords: torch.Tensor, z_coords: torch.Tensor, width_offset: torch.Tensor,
                 height_offset: torch.Tensor, map_res: float, map_height: Optional[int] = None,
                 flip_h: bool = True, device: Optional[torch.device] = None,
                 _validate_args: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
  """World x, z → integer map bins, rounding half up (maps.py:944-1019)."""
  dev = _pick_device(device, x_coords, z_coords)
  x, z, shape, b = _coords_pair(x_coords, z_coords, dev)
  if flip_h:
    assert map_height is not None
  woff = prm.upload(prm.per_sample(width_offset, b).contiguous(), dev)
  hoff = prm.upload(prm.per_sample(height_offset, b).contiguous(), dev)
  xb = torch.empty(x.shape, dtype=torch.int64, device=dev)
  zb = torch.empty(x.shape, dtype=torch.int64, device=dev)
  with torch.cuda.device(dev):
    rc = nat.lib().dm_map_quantize_f32(x.data_ptr(), z.data_ptr(), woff.data_ptr(), hoff.data_ptr(), b,
                                       x.shape[1], map_res, int(map_height or 0), int(bool(flip_h)),
                                       xb.data_ptr(), zb.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_map_quantize_f32")
  out_shape = shape if len(shape) >= 2 else (1, xb.numel())
  return xb.reshape(out_shape), zb.reshape(out_shape)


def map_dequantize(x_coords: torch.Tensor, z_coords: torch.Tensor, width_offset: torch.Tensor,
                   height_offset: torch.Tensor, map_res: float, map_height: Optional[int] = None,
                   flip_h: bool = True, device: Optional[torch.device] = None,
                   _validate_args: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
  """Inverse of map_quantize (maps.py:1021-1087)."""
  dev = _pick_device(device, x_coords, z_coords)
  xb, zb, shape, b = _coords_pair(x_coords, z_coords, dev)
  if flip_h:
    assert map_height is not None
  woff = prm.upload(prm.per_sample(width_offset, b).contiguous(), dev)
  hoff = prm.upload(prm.per_sample(height_offset, b).contiguous(), dev)
  x = torch.empty_like(xb)
  z = torch.empty_like(zb)
  with torch.cuda.device(dev):
    rc = nat.lib().dm_map_dequantize_f32(xb.data_ptr(), zb.data_ptr(), woff.data_ptr(), hoff.data_ptr(), b,
                                         xb.shape[1], map_res, int(map_height or 0), int(bool(flip_h)),
                                         x.data_ptr(), z.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_map_dequantize_f32")
  out_shape = shape if len(shape) >= 2 else (1, x.numel())
  return x.reshape(out_shape), z.reshape(out_shape)


def project(coords: torch.Tensor, values: torch.Tensor, masks: torch.Tensor, canvas: torch.Tensor,
            canvas_masks: Optional[torch.Tensor] = None, fill_value: Optional[float] = None,
            reduction: Optional[Reduction] = None, device: Optional[torch.device] = None,
            _validate_args: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
  """Scatter `values` (b, ..., n) onto `canvas` (b, ..., mh, mw) at `coords` (b, ..., n, 2) =
  [row, col]; out-of-range or masked points are dropped (maps.py:1089-1173)."""
  dev = _pick_device(device, coords, values, canvas)
  coords = utils.to_tensor(coords).to(device=dev, dtype=torch.int64)
  if coords.dim() < 3:
    coords = coords.view(1, -1, 2)
  maps_, changed = utils.scatter_tensor(canvas=canvas, indices=coords, values=values, masks=masks,
                                        fill_value=fill_value, reduction=reduction)
  if canvas_masks is not None:
    cm = utils.to_tensor(canvas_masks).to(device=dev, dtype=torch.bool)
    changed = torch.logical_or(torch.broadcast_to(cm, changed.shape), changed)
  return maps_, changed


def compute_center_offsets(cam_pose: torch.Tensor, width_offset: torch.Tensor, height_offset: torch.Tensor,
                           map_res: float, map_width: float, map_height: int, to_global: bool,
                           center_mode: CenterMode = CenterMode.none, device: Optional[torch.device] = None,
                           _validate_args: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
  """Map offsets that put the origin / the camera at the map centre (maps.py:1175-1248).
  A handful of floats per sample: host arithmetic (float32, reference op order); the results
  are host tensors that feed the kernels' parameter blocks."""
  center_mode = CenterMode(center_mode)
  pose = prm.host_f32(np.zeros(3, np.float32) if cam_pose is None else cam_pose)
  woff = prm.host_f32(0. if width_offset is None else width_offset)
  hoff = prm.host_f32(0. if height_offset is None else height_offset)
  if center_mode is CenterMode.none:
    return woff + 0., hoff + 0.
  pose = pose.reshape(-1, 3)
  center_x = torch.zeros(pose.shape[0])
  center_z = torch.zeros(pose.shape[0])
  if center_mode is CenterMode.camera and to_global:
    # local_to_global_space of the origin: rot(0) + (x, 0, z)   (maps.py:1228-1233)
    center_x = center_x + pose[:, 0]
    center_z = center_z + pose[:, 1]
  # map_quantize(width_offset=0., height_offset=0., flip_h=False)   (maps.py:1235-1243)
  res = torch.tensor(map_res, dtype=torch.float32)
  qx = torch.floor(center_x / res + 0. + 0.5).to(torch.int64).view(1, -1)
  qz = torch.floor(center_z / res + 0. + 0.5).to(torch.int64).view(1, -1)
  return woff + (map_width / 2. - qx), hoff + (map_height / 2. - qz)


# ======== MapProjector (maps.py:1252-1749) ======================================================

# name of a functional-API parameter → where MapProjector finds its default
_INTRINSIC_DEFAULTS = {"focal_x": "fx", "focal_y": "fy", "center_x": "cx", "center_y": "cy"}
_ATTR_DEFAULTS = (
  "cam_pose", "width_offset", "height_offset", "cam_pitch", "cam_height", "map_res", "map_width",
  "map_height", "trunc_depth_min", "trunc_depth_max", "trunc_height_max", "clip_border", "to_global",
  "flip_h", "fill_value", "reduction", "device", "height",
)
_OPTIONAL_DATA = ("value_map", "valid_map", "label_map", "num_classes")
_CTOR_ARGS = (
  "width", "height", "hfov", "vfov", "cam_pose", "width_offset", "height_offset", "cam_pitch", "cam_height",
  "map_res", "map_width", "map_height", "trunc_depth_min", "trunc_depth_max", "trunc_height_max",
  "clip_border", "to_global", "flip_h", "fill_value", "reduction", "device",
)
_CTOR_ARG_SET = frozenset(_CTOR_ARGS)


def _with_projector_defaults(fn):
  """Method wrapper: every argument left at None falls back to the projector's stored default
  (the reference spells this out per method as get(arg, self.arg), maps.py:1406-1749)."""
  params = list(inspect.signature(fn).parameters.values())
  names = [p.name for p in params]
  own_defaults = {p.name: p.default for p in params if p.default is not inspect.Parameter.empty}
  keep_own = {"get_height_map", "_validate_args", "center_mode", "canvas_masks", "_emit_flow"}

  def method(self, *args, **kwargs):
    if len(args) > len(names):
      raise TypeError(f"{fn.__name__}() takes at most {len(names)} positional arguments")
    call = dict(zip(names, args))
    for k, v in kwargs.items():
      if k not in names:
        raise TypeError(f"{fn.__name__}() got an unexpected keyword argument '{k}'")
      if k in call:
        raise TypeError(f"{fn.__name__}() got multiple values for argument '{k}'")
      call[k] = v
    for name in names:
      if name in keep_own:
        call.setdefault(name, own_defaults[name])
      elif call.get(name) is None:
        if name in _INTRINSIC_DEFAULTS:
          call[name] = getattr(self.cam_params, _INTRINSIC_DEFAULTS[name])
        elif name in _ATTR_DEFAULTS:
          call[name] = getattr(self, name)
        elif name in _OPTIONAL_DATA:
          call[name] = None
        elif name not in call:
          raise TypeError(f"{fn.__name__}() missing required argument: '{name}'")
    return fn(**call)

  method.__name__ = fn.__name__
  method.__doc__ = fn.__doc__
  return method


class MapProjector():
  """Stores the camera / map configuration once so the functional APIs can be called with only
  the per-frame data; per-call keyword arguments override the stored values.  Constructor
  arguments are those of the reference (maps.py:1253-1347): width, height, hfov, vfov, cam_pose
  [x, z, yaw], width_offset, height_offset, cam_pitch, cam_height, map_res, map_width, map_height,
  trunc_depth_min/max, trunc_height_max, clip_border, to_global, flip_h, fill_value (default
  -inf), reduction, device."""

  def __init__(
    self,
    width: int,
    height: int,
    hfov: float,
    vfov: Optional[float] = None,
    cam_pose: Optional[Float3D] = None,
    width_offset: Optional[float] = None,
    height_offset: Optional[float] = None,
    cam_pitch: Optional[float] = None,
    cam_height: Optional[float] = None,
    map_res: Optional[float] = None,
    map_width: Optional[int] = None,
    map_height: Optional[int] = None,
    trunc_depth_min: Optional[float] = None,
    trunc_depth_max: Optional[float] = None,
    trunc_height_max: Optional[float] = None,
    clip_border: Optional[int] = None,
    to_global: bool = False,
    flip_h: bool = True,
    fill_value: Optional[float] = NINF,
    reduction: Optional[Reduction] = None,
    device: Optional[torch.device] = None
  ):
    given = locals()
    for name in _CTOR_ARGS:
      setattr(self, name, given[name])
    self.cam_params: CameraIntrinsics = utils.get_camera_intrinsics(
      width=self.width, height=self.height, hfov=self.hfov, vfov=self.vfov)

  def clone(self, **overrides) -> "MapProjector":
    """Shallow copy with some constructor arguments replaced (None keeps the stored value),
    maps.py:1349-1404."""
    other = copy.copy(self)  # no constructor run: clones happen several times per MapBuilder step
    intrinsics_changed = False
    for name, value in overrides.items():
      if name not in _CTOR_ARG_SET:
        raise TypeError(f"clone() got unexpected keyword arguments {sorted(set(overrides) - _CTOR_ARG_SET)}")
      if value is not None:
        setattr(other, name, value)
        intrinsics_changed = intrinsics_changed or name in ("width", "height", "hfov", "vfov")
    if intrinsics_changed:
      other.cam_params = utils.get_camera_intrinsics(width=other.width, height=other.height, hfov=other.hfov,
                                                     vfov=other.vfov)
    return other

  orth_project = _with_projector_defaults(orth_project)
  camera_affine_grid = _with_projector_defaults(camera_affine_grid)
  depth_map_to_point_cloud = _with_projector_defaults(depth_map_to_point_cloud)
  height_map_to_point_cloud = _with_projector_defaults(height_map_to_point_cloud)
  image_to_camera_space = _with_projector_defaults(image_to_camera_space)
  camera_to_image_space = _with_projector_defaults(camera_to_image_space)
  camera_to_local_space = _with_projector_defaults(camera_to_local_space)
  local_to_camera_space = _with_projector_defaults(local_to_camera_space)
  local_to_global_space = _with_projector_defaults(local_to_global_space)
  global_to_local_space = _with_projector_defaults(global_to_local_space)
  map_quantize = _with_projector_defaults(map_quantize)
  map_dequantize = _with_projector_defaults(map_dequantize)
  project = _with_projector_defaults(project)
  compute_center_offsets = _with_projector_defaults(compute_center_offsets)


# ======== TopdownMap (maps.py:1753-1955) ========================================================

class TopdownMap():
  """A top-down map with its mask, height map and the projector that produced it."""

  def __init__(self, topdown_map: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None,
               height_map: Optional[torch.Tensor] = None, map_projector: Optional[MapProjector] = None,
               is_height_map: Optional[bool] = None):
    self._proj = map_projector
    self._topdown_map = topdown_map
    self._mask = mask
    self._height_map = height_map
    if is_height_map is None:  # same object ⇒ the map is its own height map (maps.py:1781-1783)
      is_height_map = (topdown_map is not None) and (topdown_map is height_map)
    self._is_height_map = is_height_map

  @property
  def is_empty(self) -> bool:
    return self._topdown_map is None

  @property
  def is_height_map(self) -> bool:
    return self._is_height_map

  @property
  def map(self) -> torch.Tensor:
    return self._topdown_map

  @property
  def topdown_map(self) -> torch.Tensor:
    return self._topdown_map

  @property
  def height_map(self) -> torch.Tensor:
    return self._topdown_map if self._is_height_map else self._height_map

  @property
  def mask(self) -> torch.Tensor:
    return self._mask

  @property
  def proj(self) -> MapProjector:
    return self._proj

  def get_camera(self) -> torch.Tensor:
    """Map coordinates (b, 2) int64 of the camera, i.e. of the local origin (maps.py:1824-1839)."""
    return self.get_coords(torch.zeros((3,), dtype=torch.float32), is_global=False).squeeze(dim=-2)

  def get_origin(self) -> torch.Tensor:
    """Map coordinates (b, 2) int64 of the global origin (maps.py:1841-1856)."""
    return self.get_coords(torch.zeros((3,), dtype=torch.float32), is_global=True).squeeze(dim=-2)

  def get_coords(self, points: torch.Tensor, is_global: bool = True) -> torch.Tensor:
    """Map coordinates (b, n, 2) int64 [x_bin, z_bin] of 3-D points (maps.py:1858-1897)."""
    points = utils.to_tensor(points)
    if points.dim() < 3:
      points = points.view(1, -1, 3)
    if self.proj.to_global and not is_global:
      points = self.proj.local_to_global_space(points=points)
    elif (not self.proj.to_global) and is_global:
      points = self.proj.global_to_local_space(points=points)
    pos_x, pos_z = self.proj.map_quantize(x_coords=points[..., 0], z_coords=points[..., 2])
    return torch.stack((pos_x, pos_z), dim=-1)

  def get_points(self, coords: torch.Tensor) -> torch.Tensor:
    """World (x, z) (b, n, 2) float32 of map coordinates (maps.py:1899-1921)."""
    coords = utils.to_tensor(coords)
    if coords.dim() < 3:
      coords = coords.view(1, -1, 2)
    pos_x, pos_z = self.proj.map_dequantize(x_coords=coords[..., 0], z_coords=coords[..., 1])
    return torch.stack((pos_x, pos_z), dim=-1)

  def select(self, center: torch.Tensor, crop_width: int, crop_height: int,
             fill_value: Optional[float] = None) -> "TopdownMap":
    """Crop (or pad) a crop_width × crop_height window around `center` (maps.py:1923-1949)."""
    return crop_topdown_map(self, center=center, crop_width=crop_width, crop_height=crop_height,
                            fill_value=fill_value, _validate_args=True)

  def select_egocentric(self, crop_width: int, crop_height: int, cam_pose: Optional[torch.Tensor] = None,
                        width_offset: Optional[torch.Tensor] = None, height_offset: Optional[torch.Tensor] = None,
                        fill_value: Optional[float] = None) -> "TopdownMap":
    """A crop_width × crop_height window per environment in its camera frame (not in the reference);
    see crop_egocentric_map."""
    return crop_egocentric_map(self, crop_width=crop_width, crop_height=crop_height, cam_pose=cam_pose,
                               width_offset=width_offset, height_offset=height_offset, fill_value=fill_value)

  def geodesic_distance(self, traversable: torch.Tensor, sources=None) -> torch.Tensor:
    """geodesic_distance over this map's grid (not in the reference).  `sources` defaults to the agent's cell as
    get_camera() defines it, computed on the host from the projector's pose and offsets (no sync when they are host
    values, as a MapBuilder world map's and a select_egocentric window's are): the distance from the agent to every
    cell in one call."""
    if sources is None:
      sources = _camera_cells(self.proj, _geodesic_grid(traversable)[0])
    return geodesic_distance(traversable, sources)

  def merge(self, *sources: List["TopdownMap"]) -> "TopdownMap":
    raise NotImplementedError


# ======== TopdownMap functional API ===============================================================

def _crop(image: torch.Tensor, center_dev: torch.Tensor, crop_h: int, crop_w: int,
          fill_value: Optional[float]) -> torch.Tensor:
  b, c, h, w = image.shape
  dev = image.device
  lib = nat.lib()
  with torch.cuda.device(dev):
    if image.dtype == torch.bool:
      out = torch.empty((b, c, crop_h, crop_w), dtype=torch.bool, device=dev)
      rc = lib.dm_crop_nearest_u8(image.data_ptr(), center_dev.data_ptr(), b, c, h, w, crop_h, crop_w,
                                  out.data_ptr(), nat.stream_ptr(dev))
    else:
      out = torch.empty((b, c, crop_h, crop_w), dtype=torch.float32, device=dev)
      rc = lib.dm_crop_nearest_f32(image.data_ptr(), center_dev.data_ptr(), b, c, h, w, crop_h, crop_w,
                                   int(fill_value is not None), 0. if fill_value is None else fill_value,
                                   out.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_crop_nearest")
  return out


def crop_topdown_map(source: TopdownMap, center: torch.Tensor, crop_width: int, crop_height: int,
                     fill_value: Optional[float] = None, mode: str = 'nearest',
                     _validate_args: bool = True) -> TopdownMap:
  """Nearest-neighbour crop of map, mask and height map around `center` (b, 2) = [x, y] in map
  pixels, exactly as the reference's pad + grid_sample formulation resamples it
  (maps.py:1959-2037); one fused kernel per tensor (csrc/dm_points.cu crop_kernel).  Unlike the
  reference, the caller's `center` tensor is not modified (maps.py:2021-2022 does, by aliasing)."""
  if mode != 'nearest':
    raise NotImplementedError("only mode='nearest' is implemented by the B200 kernels")
  proj = source.proj
  hm = source.height_map
  dev = hm.device
  center_host = prm.host_f32(center, (2,))
  b = hm.shape[0]
  center_dev = prm.upload(prm.per_sample(center_host, b, (2,), "center").contiguous(), dev)
  base = hm[:, :1] if (hm.dim() == 4 and hm.stride(1) == 0 and hm.shape[1] > 1) else hm
  height_map = _crop(base.contiguous(), center_dev, crop_height, crop_width, NINF)
  if base is not hm:
    height_map = height_map.expand(b, hm.shape[1], crop_height, crop_width)
  mask = _crop(source.mask.to(torch.bool).contiguous(), center_dev, crop_height, crop_width, False)
  topdown_map = height_map
  if not source.is_height_map:
    topdown_map = _crop(source.topdown_map.contiguous(), center_dev, crop_height, crop_width,
                        get(fill_value, proj.fill_value))
  # new offsets (maps.py:2020-2024), float32 host arithmetic
  cx, cy = center_host[:, 0].clone(), center_host[:, 1].clone()
  if proj.flip_h:
    cy = (proj.map_height - 1) - cy
  width_offset = prm.host_f32(proj.width_offset) + crop_width / 2 - cx
  height_offset = prm.host_f32(proj.height_offset) + crop_height / 2 - cy
  new_proj = proj.clone(width_offset=width_offset, height_offset=height_offset, map_width=crop_width,
                        map_height=crop_height)
  return TopdownMap(topdown_map=topdown_map, mask=mask, height_map=height_map,
                    is_height_map=source.is_height_map, map_projector=new_proj)


def crop_egocentric_map(source: TopdownMap, crop_width: int, crop_height: int, cam_pose: Optional[torch.Tensor] = None,
                        width_offset: Optional[torch.Tensor] = None, height_offset: Optional[torch.Tensor] = None,
                        fill_value: Optional[float] = None) -> TopdownMap:
  """The crop_height × crop_width window of a global-frame map that every environment sees in its own camera frame:
  centred on the agent and turned to its heading, the observation a policy reads each step (not in the reference).
  Cell (r, c) of environment i is, by definition, the composition of this module's public functions
      (lx, lz) = map_dequantize(c, r, width_offset[i], height_offset[i], map_res, crop_height, flip_h)
      (gx, gz) = local_to_global_space((lx, 0, lz), cam_pose[i])        # crop_height * crop_width points per sample
      (X, Z)   = map_quantize(gx, gz, source offsets[i], map_res, source map_height, flip_h)
  read from the source at (Z, X), bit for bit; cells outside the source get what a merge leaves in a cell nothing
  reached: `get(fill_value, proj.fill_value, NINF)` (heights of a value map: -inf; mask: False).  The window has the
  source's map_res and flip_h; with flip_h the camera's forward direction (+z local) points up.

  cam_pose (1 or b rows of x, z, yaw) defaults to source.proj.cam_pose (a MapBuilder's world map carries the pose of
  its latest step); width_offset / height_offset (1 or b values) to crop_width / 2 and crop_height / 2, which puts the
  camera where CenterMode.camera puts it in a local-frame plot; height_offset=0 puts the agent on the bottom row.
  Poses and offsets are host values uploaded with the parameter block: a CUDA pose tensor is copied to the host, which
  synchronises with its stream.  One kernel launch (csrc/dm_points.cu crop_egocentric_kernel), no host sync otherwise.

  The result's projector is source.proj.clone(cam_pose=, to_global=False, width_offset=, height_offset=,
  map_width=crop_width, map_height=crop_height), so its get_camera() is the agent's cell.  A height map stays a height
  map; a height source that is one plane expanded over the channels (a value map's local map) gives one plane,
  expanded the same way.  ValueError for an empty or local-frame source, a crop size below 1, and a pose or offset
  count other than 1 or b; all before any device work."""
  if source is None or source.is_empty:
    raise ValueError("select_egocentric needs a map: the source is empty")
  proj = source.proj
  if proj is None or not proj.to_global:
    raise ValueError("select_egocentric reads a global-frame map (proj.to_global); the source is in a local frame")
  crop_width, crop_height = int(crop_width), int(crop_height)
  if crop_width < 1 or crop_height < 1:
    raise ValueError(f"crop size must be at least 1 x 1, got {crop_width} x {crop_height}")
  top = utils.to_4D_image(source.topdown_map)
  b, C, Hs, Ws = top.shape
  pose_host = prm.host_f32(get(cam_pose, proj.cam_pose, [0., 0., 0.]), (3,))
  pose = prm.per_sample(pose_host, b, (3,), "cam_pose")
  woff = get(width_offset, crop_width / 2.)
  hoff = get(height_offset, crop_height / 2.)
  cols = [prm.per_sample(get(proj.width_offset, 0.), b, (), "source width_offset"),
          prm.per_sample(get(proj.height_offset, 0.), b, (), "source height_offset"),
          prm.per_sample(woff, b, (), "width_offset"), prm.per_sample(hoff, b, (), "height_offset")]
  dev = _pick_device(proj.device, source.mask, top)
  samples = prm.upload(prm.ego_samples(pose, *cols, crop_height * crop_width), dev)
  top = top.to(device=dev, dtype=torch.float32).contiguous()
  mask = utils.to_4D_image(source.mask).to(device=dev, dtype=torch.bool).expand(b, C, Hs, Ws).contiguous()
  out_top = torch.empty((b, C, crop_height, crop_width), dtype=torch.float32, device=dev)
  out_mask = torch.empty((b, C, crop_height, crop_width), dtype=torch.bool, device=dev)
  height = out_height = None
  plane_stride = 0
  if not source.is_height_map:
    hm = utils.to_4D_image(source.height_map).to(device=dev, dtype=torch.float32).expand(b, C, Hs, Ws)
    shared = hm.stride(1) == 0 and C > 1   # one plane for the C channels, as crop_topdown_map keeps it
    height = (hm[:, :1] if shared else hm).contiguous()
    plane_stride = 0 if shared else Hs * Ws
    out_height = torch.empty((b, 1 if shared else C, crop_height, crop_width), dtype=torch.float32, device=dev)
  fill = get(fill_value, proj.fill_value, NINF)
  with torch.cuda.device(dev):
    rc = nat.lib().dm_crop_egocentric_f32(top.data_ptr(), nat.ptr(height), plane_stride, mask.data_ptr(), b, C, Hs, Ws,
                                          float(proj.map_res), int(bool(proj.flip_h)), samples.data_ptr(),
                                          crop_height, crop_width, fill, out_top.data_ptr(), nat.ptr(out_height),
                                          out_mask.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_crop_egocentric_f32")
  if source.is_height_map:
    out_height = out_top
  elif out_height.shape[1] != C:
    out_height = out_height.expand(b, C, crop_height, crop_width)
  new_proj = proj.clone(cam_pose=pose_host, to_global=False,
                        width_offset=prm.host_f32(woff), height_offset=prm.host_f32(hoff), map_width=crop_width,
                        map_height=crop_height)
  return TopdownMap(topdown_map=out_top, mask=out_mask, height_map=out_height, is_height_map=source.is_height_map,
                    map_projector=new_proj)


def score_poses(source: TopdownMap, planes: torch.Tensor, window: torch.Tensor, cam_poses,
                width_offset=None, height_offset=None) -> torch.Tensor:
  """How well a local window matches the planes of a global-frame map at each of n candidate poses, for every
  environment at once (not in the reference): correlative scan matching, to correct noisy odometry before a merge.

  source: a global-frame TopdownMap; only its projector (map_res, flip_h, per-environment width_offset /
  height_offset) and its b x Hs x Ws size are read.  planes: CUDA bool (b, Hs, Ws) or (b, C, Hs, Ws) on the source's
  grid, what to match against (world obstacle cells, world free cells, ...).  window: CUDA bool (b, h, w), shared by
  every plane, or (b, C, h, w), one per plane (4-D planes only): the local observation, e.g. the local map's obstacle
  cells.  cam_poses: float (n, 3), shared by the environments, or (b, n, 3), rows [x, z, yaw], n >= 1.
  width_offset / height_offset (1 or b values): the window's origin, by default w / 2 and h / 2 as in
  crop_egocentric_map; a config-4 local map (to_global=False, width_offset=MW / 2, height_offset=0) passes its own.
  Returns int32 (b, n) for 3-D planes and (b, C, n) for 4-D planes.

  Definition, exact:
      score[i, c, k] = sum over (r, col) of window[i, c or 0, r, col]  AND
          crop_egocentric_map(TopdownMap(mask=planes) with source.proj, w, h, cam_pose=cam_poses[i, k],
                              width_offset, height_offset).mask[i, c, r, col]
  i.e. window cell (r, col) goes through map_dequantize with the window offsets, local_to_global_space with candidate
  k (h * w points, so the fused or naive rotation is chosen as for the crop), map_quantize with the source offsets, and
  a read of the plane there; cells that land outside the source count as False.  Integer counts: the result does not
  depend on evaluation order.  The best pose is the caller's choice, scores.argmax(-1) (the first maximum).

  Noisy-odometry recipe for a height-map MapBuilder `builder` with config-4 local maps (to_global=False,
  width_offset=MW / 2, height_offset=0), odometry poses `odom` (b, 3) on the host:
    world = builder.world_map
    seen = world.mask[:, 0]
    obstacle = seen & (world.height_map[:, 0] > obstacle_height)
    planes = torch.stack((obstacle, seen & ~obstacle), dim=1)                # world obstacle and free cells
    local = builder.plot(depth, cam_pose=odom, **config4)                    # orth_project in the camera frame
    window = local.mask[:, 0] & (local.height_map[:, 0] > obstacle_height)   # local obstacle cells
    cands = (odom[:, None, :] + lattice[None]).to(torch.float32)             # (b, n, 3): (dx, dz, dyaw) offsets
    s = score_poses(world, planes, window, cands, width_offset=MW / 2, height_offset=0.)
    best = (s[:, 0] - s[:, 1]).argmax(-1)        # obstacle hits minus local obstacles on known free cells
    pose = cands[torch.arange(b), best.cpu()]    # reading the winner back: the caller's one host sync
    builder.step(depth, cam_pose=pose, **config4)
  The read-back is the only sync the recipe adds; the growing-map MapBuilder.step already syncs once per step for
  its bounding box.

  cam_poses, like crop_egocentric_map's pose and the offsets, are host values packed into one block per (environment,
  candidate); a CUDA cam_poses tensor is copied to the host, which synchronises with its stream.  Blocks up to 64 KiB
  go through the parameter ring, larger ones through a pinned non-blocking copy: no host sync otherwise.  One library
  call on the current stream (csrc/dm_match.cu: a compaction and a scoring kernel); planes and window are never
  written.  ValueError, before any device work, for an empty or local-frame source; planes or window not bool or of
  the wrong rank; planes whose batch or Hs x Ws differs from the source; a window not (b, h, w) or (b, C, h, w), or
  with an empty dimension; cam_poses not (n, 3) or (b, n, 3) or with n < 1; an offset count other than 1 or b; b * n,
  h * w or Hs * Ws of 2^31 or more; and planes or window off CUDA or on different devices."""
  if source is None or source.is_empty:
    raise ValueError("score_poses needs a map: the source is empty")
  proj = source.proj
  if proj is None or not proj.to_global:
    raise ValueError("score_poses reads a global-frame map (proj.to_global); the source is in a local frame")
  b, _, Hs, Ws = utils.to_4D_image(source.topdown_map).shape
  for name, t in (("planes", planes), ("window", window)):
    if not torch.is_tensor(t) or t.dtype is not torch.bool:
      raise ValueError(f"{name} must be a bool tensor, got {t.dtype if torch.is_tensor(t) else type(t).__name__}")
  if planes.dim() not in (3, 4):
    raise ValueError(f"planes must be (b, Hs, Ws) or (b, C, Hs, Ws), got {tuple(planes.shape)}")
  C = planes.shape[1] if planes.dim() == 4 else 1
  if planes.shape[0] != b or tuple(planes.shape[-2:]) != (Hs, Ws) or C < 1:
    raise ValueError(f"planes must be ({b}, [C,] {Hs}, {Ws}) like the source map, got {tuple(planes.shape)}")
  per_plane = window.dim() == 4
  if not (window.dim() == 3 or (per_plane and planes.dim() == 4 and window.shape[1] == C)) or window.shape[0] != b:
    raise ValueError(f"window must be ({b}, h, w)" + (f" or ({b}, {C}, h, w)" if planes.dim() == 4 else "") +
                     f", got {tuple(window.shape)}")
  h, w = window.shape[-2], window.shape[-1]
  if h < 1 or w < 1:
    raise ValueError(f"window must not be empty, got {tuple(window.shape)}")
  pose_shape = tuple(cam_poses.shape) if torch.is_tensor(cam_poses) else np.shape(cam_poses)
  if not (len(pose_shape) == 2 or (len(pose_shape) == 3 and pose_shape[0] == b)) or pose_shape[-1] != 3 or \
     pose_shape[-2] < 1:
    raise ValueError(f"cam_poses must be (n, 3) or ({b}, n, 3) with n >= 1, got {pose_shape}")
  n = pose_shape[-2]
  for what, cells in (("b * n", b * n), ("h * w", h * w), ("Hs * Ws", Hs * Ws)):
    if cells >= 2 ** 31:
      raise ValueError(f"{what} = {cells} is too large: it must stay below 2^31")
  cols = [prm.per_sample(get(proj.width_offset, 0.), b, (), "source width_offset"),
          prm.per_sample(get(proj.height_offset, 0.), b, (), "source height_offset"),
          prm.per_sample(get(width_offset, w / 2.), b, (), "width_offset"),
          prm.per_sample(get(height_offset, h / 2.), b, (), "height_offset")]
  dev = planes.device
  if not planes.is_cuda:
    raise ValueError(f"planes must be on a CUDA device, got {dev}")
  if window.device != dev:
    raise ValueError(f"window must be on {dev}, got {window.device}")
  if torch.is_tensor(cam_poses) and cam_poses.is_cuda and cam_poses.device != dev:
    raise ValueError(f"cam_poses must be on {dev} or the host, got {cam_poses.device}")
  poses = prm.host_f32(cam_poses, (3,))
  poses = poses.reshape(-1, n, 3).expand(b, n, 3).reshape(b * n, 3)
  cols = [c[:, None].expand(b, n).reshape(b * n) for c in cols]
  samples = prm.ego_samples(poses, *cols, h * w)
  pl = planes.reshape(b, C, Hs, Ws).contiguous()
  win = window.contiguous()
  out = torch.empty((b, C, n), dtype=torch.int32, device=dev)
  with torch.cuda.device(dev):
    block = prm.upload(samples, dev) if samples.numel() * 4 <= prm._UPLOAD_MAX else \
        samples.pin_memory().to(dev, non_blocking=True)
    rc = nat.lib().dm_score_poses_i32(pl.data_ptr(), b, C, Hs, Ws, float(proj.map_res), int(bool(proj.flip_h)),
                                      win.data_ptr(), C if per_plane else 1, h, w, block.data_ptr(), n,
                                      out.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_score_poses_i32")
  return out if planes.dim() == 4 else out.view(b, n)


def _geodesic_grid(traversable) -> Tuple[int, int, int]:
  """(b, H, W) of a traversable grid, checked in every respect but its device."""
  if not torch.is_tensor(traversable) or traversable.dtype is not torch.bool:
    raise ValueError("traversable must be a bool tensor, got "
                     f"{traversable.dtype if torch.is_tensor(traversable) else type(traversable).__name__}")
  if not (traversable.dim() == 3 or (traversable.dim() == 4 and traversable.shape[1] == 1)):
    raise ValueError(f"traversable must be (b, H, W) or (b, 1, H, W), got {tuple(traversable.shape)}")
  b, H, W = traversable.shape[0], traversable.shape[-2], traversable.shape[-1]
  if b < 1 or H < 1 or W < 1:
    raise ValueError(f"traversable must not be empty, got {tuple(traversable.shape)}")
  if 7 * H * W > 2 ** 31 - 1:
    raise ValueError(f"a {H} x {W} grid is too large: its largest distance 7 * H * W does not fit in int32")
  return b, H, W


def geodesic_distance(traversable: torch.Tensor, sources) -> torch.Tensor:
  """Shortest-path distance, through traversable cells, from the sources of each environment to every cell of its map
  (not in the reference): the distance field a planner steps down, on the device, for a whole batch at once.

  traversable: CUDA bool (b, H, W) or (b, 1, H, W).  sources: a bool mask of the same shape on the same device, or
  integer cells [x, z] = [column, row] (the convention of get_coords / get_camera) of shape (b, n, 2) or (b, 2), on
  that device or on the host (host cells are uploaded through the parameter ring).  Cells outside the map are ignored.
  Returns int32 (b, H, W).

  Definition: the cells are the nodes of a graph.  An edge runs from u to an 8-neighbour v when T[v] holds and the
  step is orthogonal, or diagonal with both cells that share an edge with u and v traversable (no corner cutting).  An
  orthogonal step costs 5, a diagonal one 7.  dist[v] = 0 for a source; otherwise the least total cost of a path from
  any source of the environment, or -1 when there is none.  The distance in metres is dist * map_res / 5.
  - Integer costs make the result exact and independent of evaluation order, so it is compared bit for bit.
  - A 5 / 7 chamfer stays within about 2 % of the Euclidean length of straight paths.
  - Edges depend on the traversability of the destination only: a source cell that is an obstacle still reaches its
    free neighbours, so an object's class plane can be the goal as it is.
  Deriving `traversable` stays with the caller.  For a height world map `m` of a MapBuilder, with heights above the
  floor: `free = m.mask & (m.height_map <= obstacle_height)`, and `free | ~m.mask` when unknown cells count as free.

  One library call on the current stream (csrc/dm_geodesic.cu, one cooperative launch) and no host sync.  ValueError,
  before any device work, for another shape, dtype or device, zero source cells, and grids whose largest distance
  7 * H * W does not fit in int32."""
  b, H, W = _geodesic_grid(traversable)
  mask = cells = None
  if torch.is_tensor(sources) and sources.dtype is torch.bool:
    if sources.shape != traversable.shape:
      raise ValueError(f"a source mask must have traversable's shape {tuple(traversable.shape)}, got "
                       f"{tuple(sources.shape)}")
    mask = sources
  else:
    cells = sources if torch.is_tensor(sources) else torch.from_numpy(np.asarray(sources))
    if cells.dtype is torch.bool or cells.is_floating_point() or cells.is_complex():
      raise ValueError(f"source cells must be integers (or a bool mask), got {cells.dtype}")
    if cells.dim() == 2:
      cells = cells.unsqueeze(1)
    if cells.dim() != 3 or cells.shape[0] != b or cells.shape[2] != 2 or cells.shape[1] < 1:
      raise ValueError(f"source cells must be ({b}, n, 2) with n >= 1 or ({b}, 2), got {tuple(sources.shape)}")
  dev = traversable.device
  if not traversable.is_cuda:
    raise ValueError(f"traversable must be on a CUDA device, got {dev}")
  if mask is not None and mask.device != dev:
    raise ValueError(f"the source mask must be on {dev}, got {mask.device}")
  if cells is not None and cells.is_cuda and cells.device != dev:
    raise ValueError(f"the source cells must be on {dev} or the host, got {cells.device}")
  n = 0
  if cells is not None:
    n = cells.shape[1]
    cells = cells.to(torch.int64).contiguous()
    if not cells.is_cuda:
      cells = prm.upload(cells, dev) if cells.numel() * 8 <= prm._UPLOAD_MAX else \
          cells.pin_memory().to(dev, non_blocking=True)
  trav = traversable.reshape(b, H, W).contiguous()
  mask = None if mask is None else mask.reshape(b, H, W).contiguous()
  out = torch.empty((b, H, W), dtype=torch.int32, device=dev)
  with torch.cuda.device(dev):
    rc = nat.lib().dm_geodesic_distance_i32(trav.data_ptr(), nat.ptr(mask), nat.ptr(cells), n, b, H, W,
                                            out.data_ptr(), nat.stream_ptr(dev))
  nat.check(rc, "dm_geodesic_distance_i32")
  return out


def connected_components(mask: torch.Tensor, connectivity: int = 8, return_sizes: bool = False):
  """Connected-component labels of every H x W plane of a mask (not in the reference): frontier clusters, object
  instances of a class plane, obstacle blobs, on the device for a whole batch at once.

  mask: CUDA bool (b, H, W) or (b, C, H, W); each plane is labelled on its own, so the C class planes of a semantic map
  are C separate problems.  Non-contiguous views (world.mask[:, 0], an expanded plane) are made contiguous.
  connectivity: 4 (orthogonal neighbours) or 8 (orthogonal and diagonal neighbours).  8-connectivity has no corner rule:
  two cells that touch only at a corner are joined even when both cells beside that corner are background, so it is
  not geodesic_distance's reachability, which forbids corner cutting.  For "reachable from the agent" use
  `geodesic_distance(free, sources) >= 0`.

  Returns (labels, counts), or (labels, counts, sizes) with return_sizes=True:
  - labels: int32 with the shape of mask.  0 on background; the components of each plane are numbered 1..K in raster
    order of their first cell (the smallest row * W + col).  That is exactly scipy.ndimage.label(plane, structure)
    with structure = generate_binary_structure(2, 1) for connectivity=4 and np.ones((3, 3)) for connectivity=8.
  - counts: int32 (b,) or (b, C) on the device: K per plane.
  - sizes: int32 with the shape of mask: the cell count of each cell's component, 0 on background.  It filters by size
    without a host sync, where a per-component table would need K on the host.

  Frontier clusters of a MapBuilder world map `m` (seen free cells next to unseen ones), dropping clusters below k
  cells:
    seen = m.mask[:, 0]
    free = seen & (m.height_map[:, 0] <= obstacle_height)
    unseen_near = torch.nn.functional.max_pool2d((~seen).float()[:, None], 3, 1, 1)[:, 0] > 0
    frontier = free & unseen_near
    labels, counts, sizes = connected_components(frontier, return_sizes=True)
    labels = labels * (sizes >= k)

  One library call on the current stream (csrc/dm_components.cu: a block-based union-find in a few kernels and a cub
  scan), no host sync, mask never written.  ValueError, before any device work, for a non-tensor or non-bool mask, a
  rank other than 3 or 4, an empty dimension, a mask off CUDA, connectivity not 4 or 8, and more than 2^31 - 1 cells."""
  if not torch.is_tensor(mask) or mask.dtype is not torch.bool:
    raise ValueError("mask must be a bool tensor, got "
                     f"{mask.dtype if torch.is_tensor(mask) else type(mask).__name__}")
  if mask.dim() not in (3, 4):
    raise ValueError(f"mask must be (b, H, W) or (b, C, H, W), got {tuple(mask.shape)}")
  if mask.numel() == 0:
    raise ValueError(f"mask must not be empty, got {tuple(mask.shape)}")
  if mask.numel() > 2 ** 31 - 1:
    raise ValueError(f"a mask of {mask.numel()} cells is too large: at most 2^31 - 1 cells are labelled in one call")
  if isinstance(connectivity, bool) or connectivity not in (4, 8):
    raise ValueError(f"connectivity must be 4 or 8, got {connectivity!r}")
  if not mask.is_cuda:
    raise ValueError(f"mask must be on a CUDA device, got {mask.device}")
  H, W = mask.shape[-2], mask.shape[-1]
  dev = mask.device
  m = mask.contiguous()
  labels = torch.empty(mask.shape, dtype=torch.int32, device=dev)
  counts = torch.empty(mask.shape[:-2], dtype=torch.int32, device=dev)
  sizes = torch.empty(mask.shape, dtype=torch.int32, device=dev) if return_sizes else None
  with torch.cuda.device(dev):
    rc = nat.lib().dm_connected_components_i32(m.data_ptr(), m.numel() // (H * W), H, W, int(connectivity),
                                               labels.data_ptr(), counts.data_ptr(), nat.ptr(sizes),
                                               nat.stream_ptr(dev))
  nat.check(rc, "dm_connected_components_i32")
  return (labels, counts, sizes) if return_sizes else (labels, counts)


def distance_transform(mask: torch.Tensor, return_indices: bool = False):
  """Exact Euclidean distance transform of every H x W plane of a mask (not in the reference): the clearance of each
  cell from the nearest obstacle, and the nearest free cell to a goal, on the device for a whole batch at once.

  mask: CUDA bool (b, H, W) or (b, C, H, W); each plane is transformed on its own.  Non-contiguous views
  (world.mask[:, 0], an expanded plane) are made contiguous.

  Returns dist, or (dist, nearest) with return_indices=True:
  - dist: float32 with the shape of mask.  0 on False cells; on True cells the Euclidean distance in cells (centre to
    centre) to the nearest False cell of the same plane; in metres, dist * map_res.  That is exactly
    scipy.ndimage.distance_transform_edt(plane).astype(np.float32).
  - nearest: int32 of shape (*mask.shape, 2) holding [x, z] = [column, row], the cell convention of get_coords /
    get_camera / geodesic_distance's source cells.  It is not scipy's return_indices layout, which is (2, H, W) in
    [row, column] order.  On a True cell: a False cell at exactly the returned distance; on a False cell: the cell
    itself.  When several False cells are equally near, it is one of them, fixed: the same input gives the same bits
    on every call, and a plane's result does not depend on the other planes.  It need not be scipy's choice.
  A plane with no False cell has no nearest one: dist is +inf and nearest is -1 on every cell of it (scipy instead
  measures to a phantom cell outside the plane).

  Obstacle inflation for a MapBuilder world map `m` and an agent of radius r metres: the cells where the agent's centre
  keeps more than r from every obstacle, and the geodesic field over them:
    seen = m.mask[:, 0]
    obstacle = seen & (m.height_map[:, 0] > obstacle_height)
    free = seen & ~obstacle
    traversable = free & (distance_transform(~obstacle) * map_res > r)
    dist_to_agent = m.geodesic_distance(traversable)

  Goal snapping, the free cell nearest to goal cell (x, z) of environment i (an object goal on an obstacle, a frontier
  cell):
    d, nearest = distance_transform(~free, return_indices=True)
    x_free, z_free = nearest[i, z, x]

  One library call on the current stream (csrc/dm_distance.cu: the separable exact transform in two kernels), no host
  sync, mask never written.  ValueError, before any device work, for a non-tensor or non-bool mask, a rank other than 3
  or 4, an empty dimension, a mask off CUDA, H or W above 32768 (the squared distance must fit in int32), and more than
  2^31 - 1 cells."""
  if not torch.is_tensor(mask) or mask.dtype is not torch.bool:
    raise ValueError("mask must be a bool tensor, got "
                     f"{mask.dtype if torch.is_tensor(mask) else type(mask).__name__}")
  if mask.dim() not in (3, 4):
    raise ValueError(f"mask must be (b, H, W) or (b, C, H, W), got {tuple(mask.shape)}")
  if mask.numel() == 0:
    raise ValueError(f"mask must not be empty, got {tuple(mask.shape)}")
  H, W = mask.shape[-2], mask.shape[-1]
  if H > 32768 or W > 32768:
    raise ValueError(f"a {H} x {W} plane is too large: H and W must be at most 32768 so that the squared distance fits "
                     "in int32")
  if mask.numel() > 2 ** 31 - 1:
    raise ValueError(f"a mask of {mask.numel()} cells is too large: at most 2^31 - 1 cells are transformed in one call")
  if not mask.is_cuda:
    raise ValueError(f"mask must be on a CUDA device, got {mask.device}")
  dev = mask.device
  m = mask.contiguous()
  dist = torch.empty(mask.shape, dtype=torch.float32, device=dev)
  nearest = torch.empty((*mask.shape, 2), dtype=torch.int32, device=dev) if return_indices else None
  with torch.cuda.device(dev):
    rc = nat.lib().dm_distance_transform_f32(m.data_ptr(), m.numel() // (H * W), H, W, dist.data_ptr(),
                                             nat.ptr(nearest), nat.stream_ptr(dev))
  nat.check(rc, "dm_distance_transform_f32")
  return (dist, nearest) if return_indices else dist


def _camera_cells(proj: MapProjector, b: int) -> torch.Tensor:
  """TopdownMap.get_camera() of b environments, (b, 2) int64 [x, z], from the projector's host values: the local
  origin, moved by local_to_global_space for a global-frame map ((0, 0, 0) rotated is +-0, so it lands on the pose's
  x, z exactly), then map_quantize in the same float32 operations."""
  zero = torch.zeros((b,), dtype=torch.float32)
  x = z = zero
  if proj.to_global:
    pose = prm.per_sample(prm.host_f32(get(proj.cam_pose, [0., 0., 0.]), (3,)), b, (3,), "cam_pose")
    x, z = pose[:, 0] + zero, pose[:, 1] + zero
  res = torch.tensor(float(proj.map_res), dtype=torch.float32)
  xb = x / res + prm.per_sample(get(proj.width_offset, 0.), b, (), "width_offset")
  zb = z / res + prm.per_sample(get(proj.height_offset, 0.), b, (), "height_offset")
  if proj.flip_h:
    zb = torch.tensor(float(proj.map_height - 1), dtype=torch.float32) - zb
  return torch.stack((torch.floor(xb + 0.5), torch.floor(zb + 0.5)), dim=-1).to(torch.int64)


def _fuse_source(m: TopdownMap, target: MapProjector, b: int, C: int, n_total: int, dev: torch.device,
                 keep: list) -> nat.DmFuseSource:
  hm = m.height_map.to(device=dev, dtype=torch.float32)
  if hm.dim() != 4:
    hm = utils.to_4D_image(hm)
  h, w = hm.shape[-2:]
  if hm.stride(-1) != 1 or hm.stride(-2) != w:
    hm = hm.contiguous()
  hm = hm.expand(b, C, h, w)
  mask = m.mask.to(device=dev, dtype=torch.bool).expand(b, C, h, w).contiguous()
  values = None
  if not m.is_height_map:
    values = m.topdown_map.to(device=dev, dtype=torch.float32).expand(b, C, h, w).contiguous()
  pose = prm.per_sample(get(m.proj.cam_pose, [0., 0., 0.]), b, (3,), "cam_pose")
  tpose = prm.per_sample(get(target.cam_pose, [0., 0., 0.]), b, (3,), "cam_pose")
  # maps.py:2059-2060: a local map goes to global space with its own pose;
  # maps.py:2116-2117: everything goes to the target's local space if the target is local
  s0 = prm.identity(b) if m.proj.to_global else prm.local_to_global(pose, C * h * w)
  s1 = prm.identity(b) if target.to_global else prm.global_to_local(tpose, n_total)
  # one parameter block per source: [steps (b, 2, 16 words) | width offsets (b,) | height offsets (b,)], one upload
  params = torch.cat((torch.cat((s0, s1), dim=1).reshape(-1),
                      prm.per_sample(get(m.proj.width_offset, 0.), b).reshape(-1),
                      prm.per_sample(get(m.proj.height_offset, 0.), b).reshape(-1)))
  params_dev = prm.upload(params, dev)
  n_step_words = b * 2 * prm.STEP_WORDS
  keep.extend((hm, mask, values, params_dev))
  src = nat.DmFuseSource()
  src.height, src.values, src.mask = hm.data_ptr(), nat.ptr(values), mask.data_ptr()
  src.height_bstride, src.height_cstride = hm.stride(0), hm.stride(1)
  src.h, src.w = h, w
  src.flip_h = bool(m.proj.flip_h)
  src.map_res = m.proj.map_res
  base = params_dev.data_ptr()
  src.steps, src.width_offset, src.height_offset = base, base + 4 * n_step_words, base + 4 * (n_step_words + b)
  # a map this module wrote carries, per plane, the rectangle that holds its valid cells: the passes scan that instead
  # of the whole plane (a grown world map is mostly empty canvas)
  planes = _tracked_planes(m, dev, b * C)
  if planes is not None:
    src.plane_box = planes.data_ptr()
    keep.append(planes)
  return src


def fuse_topdown_maps(*maps: List[TopdownMap], map_projector: Optional[MapProjector] = None,
                      fill_value: Optional[float] = None, reduction: Optional[Reduction] = None) -> TopdownMap:
  """Re-project several top-down maps into one freshly sized map in `map_projector`'s frame
  (maps.py:2181-2287): every valid cell becomes a point again, one bounding box over all of them
  sizes the canvas (host sync), and the points are scatter-maxed into it.  Two fused passes over
  the source cells (csrc/dm_fuse.cu), no point cloud is materialised."""
  if len(maps) == 0:
    return TopdownMap(map_projector=map_projector)
  proj = map_projector if map_projector is not None else maps[0].proj
  live = [m for m in maps if not m.is_empty]
  if not live:
    return TopdownMap(map_projector=proj)
  kinds = {bool(m.is_height_map) for m in live}
  assert len(kinds) == 1, "All maps must be the same type of maps (all height maps or all value maps)."
  is_height_map = kinds.pop()
  # MapProjector.project: get(reduction, self.reduction), maps.py:1720.  All five reductions: max / min through the
  # atomic scatter, sum / mean / prod through the ordered fold (csrc/dm_ordered.cu: the reference's point order)
  red = utils._reduction_code(get(reduction, proj.reduction), fused=False)
  dev = _pick_device(proj.device, *[m.mask for m in live], *[m.height_map for m in live])
  shapes = [utils.to_4D_image(m.mask).shape for m in live]
  b = max(s[0] for s in shapes)
  C = max(s[1] for s in shapes)
  n_total = sum(C * s[2] * s[3] for s in shapes)
  keep: list = []
  # A map that an earlier call of this function produced carries the bounding box pass 1 would find for it
  # (_TrackedBox); it then only seeds the box and pass 1 scans the other maps — for a MapBuilder that is the local
  # map instead of the whole world map, ahead of the host sync below.
  seed = next((m for m in live if _tracked_box_valid(m, proj, dev)), None)
  scan = [m for m in live if m is not seed]
  all_sources = [_fuse_source(m, proj, b, C, n_total, dev, keep) for m in live]
  sources = (nat.DmFuseSource * len(live))(*all_sources)
  scan_sources = (nat.DmFuseSource * max(len(scan), 1))(*[s for m, s in zip(live, all_sources) if m is not seed])
  lib = nat.lib()
  bbox = torch.empty((5,), dtype=torch.int64, device=dev)
  with torch.cuda.device(dev):
    rc = lib.dm_fuse_bbox_seeded_i64(scan_sources, len(scan), b, C, proj.map_res,
                                     None if seed is None else seed._tracked_box.box.data_ptr(), bbox.data_ptr(),
                                     nat.stream_ptr(dev))
  nat.check(rc, "dm_fuse_bbox_seeded_i64")
  min_x, max_x, min_z, max_z, n_valid = (int(v) for v in bbox.cpu())  # the reference's .item() sync
  if n_valid == 0:  # maps.py:2217-2225
    last = maps[-1]
    return TopdownMap(topdown_map=last.topdown_map, mask=last.mask, height_map=last.height_map, map_projector=proj)
  # maps.py:2171-2178 (float32 host arithmetic; exact for any realistic map size)
  map_width = (max_x - min_x) + 2
  map_height = (max_z - min_z) + 2
  # shape (1,) like the reference's (the bbox is reduced over a (1, n) view, maps.py:2159-2169)
  width_offset = torch.tensor(map_width / 2., dtype=torch.float32) - torch.tensor([max_x + min_x]) / 2.
  height_offset = torch.tensor(map_height / 2., dtype=torch.float32) - torch.tensor([max_z + min_z]) / 2.
  tgt = nat.DmFuseTarget()
  tgt.Mh, tgt.Mw = map_height, map_width
  tgt.flip_h = bool(proj.flip_h)
  tgt.map_res = proj.map_res
  tgt.width_offset, tgt.height_offset = float(width_offset), float(height_offset)
  tgt.fill_value = get(fill_value, proj.fill_value, NINF)
  tgt.reduction = red
  topdown = _alloc_canvas((b, C, map_height, map_width), torch.float32, dev)
  mask = _alloc_canvas((b, C, map_height, map_width), torch.bool, dev)
  height = None if is_height_map else _alloc_canvas((b, C, map_height, map_width), torch.float32, dev)
  # the new map is in the global frame when the target is: pass 2 then leaves its box for the next merge
  track = bool(proj.to_global) and tgt.fill_value == tgt.fill_value and red < 2
  next_box = torch.empty((5,), dtype=torch.int64, device=dev) if track else None
  # ... and, whatever the frame, the per-plane rectangles of its valid cells (cell coordinates: no projector involved)
  track_planes = tgt.fill_value == tgt.fill_value and red < 2
  plane_box = torch.empty((b * C, 4), dtype=torch.int32, device=dev) if track_planes else None
  with torch.cuda.device(dev):
    rc = lib.dm_fuse_scatter_track_f32(sources, len(live), b, C, tgt, topdown.data_ptr(), mask.data_ptr(),
                                       nat.ptr(height), nat.ptr(next_box), nat.ptr(plane_box), nat.stream_ptr(dev))
  nat.check(rc, "dm_fuse_scatter_track_f32")
  new_proj = proj.clone(width_offset=width_offset, height_offset=height_offset, map_width=map_width,
                        map_height=map_height)
  out = TopdownMap(topdown_map=topdown, mask=mask, height_map=topdown if is_height_map else height,
                   map_projector=new_proj, is_height_map=is_height_map)
  if track or track_planes:
    out._tracked_box = _TrackedBox(next_box, mask, new_proj, plane_box)
  return out


class _TrackedBox():
  """Bounding box (device, 5 x int64) that pass 1 of fuse_topdown_maps would compute for a map this module wrote,
  with what it was derived from: the mask tensor (and its in-place version counter) and the projector's
  dequantisation parameters.  Anything that no longer matches makes the map an ordinary, scanned source again."""

  def __init__(self, box: Optional[torch.Tensor], mask: torch.Tensor, proj: MapProjector,
               plane_box: Optional[torch.Tensor] = None):
    self.box = box              # None: only the per-plane rectangles are tracked (local-frame target)
    self.plane_box = plane_box  # (b*C, 4) int32 device: rows [min, max], columns [min, max] of every plane's valid cells
    self.mask = mask
    self.mask_version = mask._version
    self.proj = proj
    self.key = self.proj_key(proj)

  @staticmethod
  def proj_key(proj: MapProjector):
    f = lambda x: None if x is None else tuple(float(v) for v in torch.as_tensor(x).reshape(-1))
    return (f(proj.width_offset), f(proj.height_offset), float(proj.map_res), bool(proj.flip_h), bool(proj.to_global))


def _tracked_box_valid(m: TopdownMap, target: MapProjector, dev: torch.device) -> bool:
  tb = getattr(m, "_tracked_box", None)
  if tb is None or tb.box is None or not target.to_global:
    return False
  return (m.mask is tb.mask and tb.mask._version == tb.mask_version and tb.box.device == dev
          and m.proj is tb.proj and tb.proj_key(m.proj) == tb.key and tb.key[4]
          and float(target.map_res) == tb.key[2])


def _tracked_planes(m: TopdownMap, dev: torch.device, n_planes: int) -> Optional[torch.Tensor]:
  """The per-plane rectangles m carries (_TrackedBox.plane_box) while they still describe its mask: the same mask
  tensor at the same version, rectangles on `dev`, one row for each of n_planes planes.  Else None."""
  tb = getattr(m, "_tracked_box", None)
  if (tb is None or tb.plane_box is None or m.mask is not tb.mask or tb.mask._version != tb.mask_version
      or tb.plane_box.device != dev or tb.plane_box.shape[0] != n_planes):
    return None
  return tb.plane_box


def merge_into_canvas(world: TopdownMap, new_map: TopdownMap, canvas_shape: Tuple[int, int],
                      map_projector: MapProjector, fill_value: Optional[float] = None,
                      reduction: Optional[Reduction] = None) -> TopdownMap:
  """Opt-in fixed-canvas merge (not in the reference; its closest relative is project(..., canvas=,
  canvas_masks=), maps.py:1089-1173): the valid cells of `new_map` become points again exactly as in
  fuse_topdown_maps (dequantise, local → global with the map's own pose), are quantised with the
  canvases' FIXED offsets (map_width / 2, map_height / 2: world origin at the centre) and max-merged in
  place into `world`'s tensors, which are allocated on the first call.  One launch, no host sync.
  `world`'s tensors are updated in place and shared with the returned map."""
  Hc, Wc = int(canvas_shape[0]), int(canvas_shape[1])
  red = utils._reduction_code(get(reduction, map_projector.reduction), fused=False)
  if new_map.is_empty:
    return world
  dev = _pick_device(map_projector.device, new_map.mask, new_map.height_map)
  b, C, _, _ = utils.to_4D_image(new_map.mask).shape
  is_height_map = bool(new_map.is_height_map)
  fill = get(fill_value, map_projector.fill_value, NINF)
  lib = nat.lib()
  if world is None or world.is_empty:
    topdown = torch.empty((b, C, Hc, Wc), dtype=torch.float32, device=dev)
    mask = torch.empty((b, C, Hc, Wc), dtype=torch.bool, device=dev)
    height = None if is_height_map else torch.empty_like(topdown)
    with torch.cuda.device(dev):
      rc = lib.dm_fuse_canvas_init_f32(topdown.data_ptr(), mask.data_ptr(), nat.ptr(height), topdown.numel(),
                                       fill, nat.stream_ptr(dev))
    nat.check(rc, "dm_fuse_canvas_init_f32")
  else:
    assert bool(world.is_height_map) == is_height_map, "All maps must be the same type of maps"
    topdown, mask = world.topdown_map, world.mask
    height = None if is_height_map else world.height_map
    assert tuple(topdown.shape) == (b, C, Hc, Wc), f"world canvas {tuple(topdown.shape)} != {(b, C, Hc, Wc)}"
  target = map_projector.clone(to_global=True, width_offset=Wc / 2., height_offset=Hc / 2., map_width=Wc,
                               map_height=Hc)
  keep: list = []
  h, w = new_map.mask.shape[-2:]
  sources = (nat.DmFuseSource * 1)(_fuse_source(new_map, target, b, C, C * h * w, dev, keep))
  tgt = nat.DmFuseTarget()
  tgt.Mh, tgt.Mw = Hc, Wc
  tgt.flip_h = bool(target.flip_h)
  tgt.map_res = target.map_res
  tgt.width_offset, tgt.height_offset = Wc / 2., Hc / 2.
  tgt.fill_value = fill
  tgt.reduction = red
  with torch.cuda.device(dev):
    rc = lib.dm_fuse_inplace_f32(sources, 1, b, C, tgt, topdown.data_ptr(), mask.data_ptr(), nat.ptr(height),
                                 nat.stream_ptr(dev))
  nat.check(rc, "dm_fuse_inplace_f32")
  return TopdownMap(topdown_map=topdown, mask=mask, height_map=topdown if is_height_map else height,
                    map_projector=target, is_height_map=is_height_map)


# ======== MapBuilder (maps.py:2289-2550) ==========================================================

class _NativeBuilder():
  """Owner of one DmBuilder handle (csrc/dm_builder.cu): a MapBuilder's step configuration frozen into C.  A height-map
  handle (C = 0) takes dm_builder_plot_prefill / _merge / _step_fixed and DmMapRef, a value-map handle the *_values
  entries and DmValueMapRef; the methods below are the one place that tells the two apart.  A map's canvases travel as
  (topdown, mask), with a value map's heights third."""

  def __init__(self, proj: MapProjector, key: tuple, dev: torch.device):
    (b, H, W, _, plot_global, woff, hoff, Mw, Mh, pitch, camh, res, _, _, tdmin, tdmax, thmax, clip, flip, fill,
     red, kind, C) = key
    self.handle = None
    cfg = nat.DmBuilderCfg()
    p = cfg.proj
    p.H, p.W, p.C, p.Mh, p.Mw = H, W, C, Mh, Mw
    k = proj.cam_params
    p.fx, p.fy, p.cx, p.cy = k.fx, k.fy, k.cx, k.cy
    p.map_res = res
    p.has_trunc_depth_min, p.has_trunc_depth_max = tdmin is not None, tdmax is not None
    p.has_trunc_height_max = thmax is not None
    p.trunc_depth_min, p.trunc_depth_max, p.trunc_height_max = tdmin or 0., tdmax or 0., thmax or 0.
    p.clip_border = int(clip) if clip is not None else 0
    p.flip_h = flip
    p.fill_value = 0. if fill is None else fill      # utils.py:472-473
    p.reduction = red
    cfg.b, cfg.plot_to_global = b, plot_global
    R = prm.rotation_matrices([1., 0., 0.], torch.tensor([pitch], dtype=torch.float32))  # maps.py:789-793
    cfg.pitch_R[:] = [float(v) for v in R.reshape(-1)]
    cfg.cam_height = camh
    cfg.width_offset, cfg.height_offset = woff, hoff
    skew, skew_sq, _ = prm._skew_terms([0., 1., 0.])
    cfg.yaw_skew[:] = [float(v) for v in skew.reshape(-1)]
    cfg.yaw_skew_sq[:] = [float(v) for v in skew_sq.reshape(-1)]
    self.fill = get(fill, NINF)                       # maps.py:2246: get(fill_value, proj.fill_value, NINF)
    cfg.merge_fill_value = self.fill
    cfg.merge_reduction = red
    self.C = C
    self.dtypes = (torch.float32, torch.bool) + ((torch.float32,) if C else ())  # of the canvases
    self._lib = nat.lib()
    handle = nat.ctypes.c_void_p()
    with torch.cuda.device(dev):
      if kind == "height":
        nat.check(self._lib.dm_builder_create(cfg, dev.index, nat.ctypes.byref(handle)), "dm_builder_create")
      else:
        nat.check(self._lib.dm_builder_create_values(cfg, int(kind == "labels"), dev.index, nat.ctypes.byref(handle)),
                  "dm_builder_create_values")
    self.handle = handle

  def canvases(self, m: TopdownMap) -> tuple:
    return (m.topdown_map, m.mask) + ((m.height_map,) if self.C else ())

  def map_ref(self, canvases, h: int, w: int, width_offset: float, height_offset: float, box=None, planes=None):
    """The DmMapRef / DmValueMapRef of (h, w) `canvases` with these offsets and tracked boxes (None: not tracked)."""
    top, mask = canvases[0].data_ptr(), canvases[1].data_ptr()
    if self.C == 0:
      return nat.DmMapRef(top, mask, h, w, width_offset, height_offset, nat.ptr(box), nat.ptr(planes))
    return nat.DmValueMapRef(top, canvases[2].data_ptr(), mask, h, w, width_offset, height_offset, nat.ptr(box),
                             nat.ptr(planes))

  def inputs(self, depth, values, labels, pose, sin, cos, local) -> tuple:
    """The leading arguments of plot() and step_fixed(): the frame, the poses with the sin / cos of their yaws, and
    the local map's canvases (a value map's with its one height plane)."""
    if self.C == 0:
      return (depth.data_ptr(), pose.data_ptr(), sin.data_ptr(), cos.data_ptr(), local[0].data_ptr(),
              local[1].data_ptr())
    return (depth.data_ptr(), nat.ptr(values), nat.ptr(labels), pose.data_ptr(), sin.data_ptr(), cos.data_ptr(),
            local[0].data_ptr(), local[1].data_ptr(), local[2].data_ptr())

  def plot(self, inputs: tuple, world, spec: Optional[list], n_guess: int, stream: int) -> None:
    """Queues the projection, the bounding box's reduction and copy, and the fill of the first n_guess cells of the
    speculative canvases `spec` (None: none); wait() blocks for the box."""
    top, mask, *height = [nat.ptr(t) for t in spec] if spec is not None else [None] * len(self.dtypes)
    lib = nat.lib()
    if self.C == 0:
      nat.check(lib.dm_builder_plot_prefill(self.handle, *inputs, world, None, top, mask, n_guess, stream),
                "dm_builder_plot_prefill")
    else:
      nat.check(lib.dm_builder_plot_values(self.handle, *inputs, world, None, top, *height, mask, n_guess, stream),
                "dm_builder_plot_values")

  def wait(self) -> "nat.DmMergeShape":
    shape = nat.DmMergeShape()
    nat.check(nat.lib().dm_builder_plot_wait(self.handle, shape), "dm_builder_plot_wait")
    return shape

  def merge(self, out, stream: int) -> None:
    if self.C == 0:
      nat.check(nat.lib().dm_builder_merge(self.handle, out, stream), "dm_builder_merge")
    else:
      nat.check(nat.lib().dm_builder_merge_values(self.handle, out, stream), "dm_builder_merge_values")

  def step_fixed(self, inputs: tuple, canvas, stream: int) -> None:
    if self.C == 0:
      nat.check(nat.lib().dm_builder_step_fixed(self.handle, *inputs, canvas, stream), "dm_builder_step_fixed")
    else:
      nat.check(nat.lib().dm_builder_step_fixed_values(self.handle, *inputs, canvas, stream),
                "dm_builder_step_fixed_values")

  def close(self):
    """Destroys the handle (dm_builder_destroy synchronises with the work it queued)."""
    if self.handle:
      self._lib.dm_builder_destroy(self.handle)
      self.handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass


class MapBuilder():
  """Plots a local top-down map per frame and merges it into a growing world map."""

  def __init__(self, map_projector: MapProjector, world_map: Optional[TopdownMap] = None,
               fixed_canvas: Optional[Tuple[int, int]] = None, native_step: bool = True):
    """`fixed_canvas=(map_height, map_width)` opts into the in-place world map (not in the reference,
    SURVEY.md §8f-2): global canvases of that size are allocated at the first merge, the world origin sits
    at their centre, and every merge max-merges the new map's cells into them with one kernel launch —
    no bounding box, no host sync, no reallocation.  Points that fall outside the canvas are dropped.
    `native_step`: steps of a global-frame builder (valid_map None, CenterMode.none, device depth tensors; height
    maps, CUDA float32 `value_map=` planes or CUDA `label_map=` class ids, reduction max / min) run with their host
    side in C (dm_builder_*, csrc/dm_builder.cu) — same kernels, same results, two library calls per step instead of
    ~1000 interpreter calls; anything else takes the general path.  Memory: while the host waits for the bounding box,
    the C step fills canvases of the old world map's size class (values, heights and mask for value maps: up to
    1.25 x the old map).  They become the new map.  When the new map outgrows them, they are released before the new
    map's canvases are taken, so the step holds at most the old map plus one canvas set of the new map's size class,
    as the general path does."""
    self._proj = map_projector
    self._world_map = world_map if world_map is not None else TopdownMap(map_projector=self.proj.clone())
    self._fixed = None if fixed_canvas is None else (int(fixed_canvas[0]), int(fixed_canvas[1]))
    self._native = bool(native_step)
    self._handles: Dict[tuple, "_NativeBuilder"] = {}  # least recently used first, at most _MAX_HANDLES
    # the mask of the world map when its canvases are the builder's own (a merge allocated them), else None:
    # reset_envs writes into those only
    self._owned: Optional[torch.Tensor] = None

  @property
  def proj(self) -> MapProjector:
    return self._proj

  @property
  def world_map(self) -> TopdownMap:
    return self._world_map

  def reset(self, depth_map: Optional[np.ndarray] = None, value_map: Optional[np.ndarray] = None,
            valid_map: Optional[np.ndarray] = None, cam_pose: Optional[np.ndarray] = None,
            center_mode: CenterMode = CenterMode.none, **kwargs):
    """Forget the world map; if a frame is given, plot and merge it (maps.py:2312-2355)."""
    self._world_map = TopdownMap(map_projector=self.proj.clone())
    self._owned = None
    if depth_map is None:
      return None
    return self.step(depth_map=depth_map, value_map=value_map, valid_map=valid_map, cam_pose=cam_pose,
                     center_mode=center_mode, **kwargs)

  def reset_envs(self, done, fill_value: Optional[float] = None) -> None:
    """Forget the world map of every environment i with done[i] set and keep the others bit for bit (not in the
    reference, whose MapBuilder is not batched): a vectorised loop whose episodes end at different steps keeps one
    batched builder.

    `done`: (b,) bools, b the world map's batch.  A CUDA bool tensor on the world map's device is read by the kernel
    only (no host sync); a CPU tensor, numpy array or list is uploaded.  ValueError for another length, another dtype
    or another CUDA device.

    Every plane of a done environment becomes what a fresh canvas holds: `get(fill_value, proj.fill_value, NINF)`
    (merge's fill rule), heights -inf (value maps; a height map's heights are its values and get the fill), mask False.
    Shape, offsets and projector stay; the next merge sizes the canvas from the cells that are left, as every merge
    does, so the map may shrink.  The per-plane rectangles and the bounding box the world map carries are kept up to
    date on the device, so the next step still starts from the box instead of scanning the world map.

    In place when the canvases are the builder's own: a world map a merge allocated, or a fixed canvas the builder
    allocated.  A world map that shares tensors with the caller (one passed to the constructor, or a local map that a
    merge adopted because nothing was valid before) is replaced by a cleared copy; the caller's tensors stay as they
    were.  With no world map yet there is nothing to do."""
    world = self._world_map
    if world is None or world.is_empty:
      return
    in_place = world.mask is self._owned
    top, mask, hm = world.topdown_map, world.mask, world.height_map
    dev = mask.device if in_place else _pick_device(self.proj.device, mask, top)
    b, C = utils.to_4D_image(mask).shape[:2]
    done_dev = self._done_flags(done, b, dev)
    fill = get(fill_value, self.proj.fill_value, NINF)
    red = utils._reduction_code(self.proj.reduction, fused=False)
    proj = world.proj if world.proj is not None else self.proj
    tb = getattr(world, "_tracked_box", None)
    planes = _tracked_planes(world, dev, b * C)
    box = tb.box if planes is not None and _tracked_box_valid(world, proj, dev) else None
    track = planes is not None and fill == fill and red < 2   # the rectangles assume "mask = beats the merge's fill"
    if not in_place:
      copy = lambda t, dt: utils.to_4D_image(t).to(device=dev, dtype=dt).clone(memory_format=torch.contiguous_format)
      top, mask = copy(top, torch.float32), copy(mask, torch.bool)
      hm = top if world.is_height_map else copy(hm, torch.float32)
      if track:
        planes, box = planes.clone(), None if box is None else box.clone()
    tgt = nat.DmFuseTarget()
    tgt.Mh, tgt.Mw = mask.shape[-2], mask.shape[-1]
    tgt.flip_h, tgt.map_res = bool(proj.flip_h), float(proj.map_res)
    if track and box is not None:
      tgt.width_offset, tgt.height_offset = float(proj.width_offset), float(proj.height_offset)
    tgt.fill_value, tgt.reduction = fill, red
    with torch.cuda.device(dev):
      rc = nat.lib().dm_fuse_clear_envs_f32(top.data_ptr(), None if world.is_height_map else hm.data_ptr(),
                                            mask.data_ptr(), b, C, done_dev.data_ptr(), tgt,
                                            nat.ptr(planes) if track else None, nat.ptr(box) if track else None,
                                            nat.stream_ptr(dev))
    nat.check(rc, "dm_fuse_clear_envs_f32")
    if not in_place:
      world = TopdownMap(topdown_map=top, mask=mask, height_map=hm, map_projector=world.proj,
                         is_height_map=world.is_height_map)
      self._world_map, self._owned = world, mask
    if track:
      world._tracked_box = _TrackedBox(box, mask, proj, planes)
    elif in_place and tb is not None:
      world._tracked_box = None   # rectangles that the clear did not update no longer describe the mask

  @staticmethod
  def _done_flags(done, b: int, dev: torch.device):
    """reset_envs' `done` as a device buffer of b bytes (0 / 1); a CUDA tensor is used as it is, unread."""
    if torch.is_tensor(done):
      if done.dtype is not torch.bool or tuple(done.shape) != (b,):
        raise ValueError(f"done must be a ({b},) bool tensor, got {done.dtype} {tuple(done.shape)}")
      if done.is_cuda:
        if done.device != dev:
          raise ValueError(f"done is on {done.device}, the world map on {dev}")
        return done.contiguous()
      return prm.upload(done.detach(), dev)
    flags = np.asarray(done)
    if flags.dtype != np.bool_ or flags.shape != (b,):
      raise ValueError(f"done must be {b} bools, got {flags.dtype} {flags.shape}")
    return prm.upload(torch.from_numpy(np.ascontiguousarray(flags)), dev)

  def step(self, depth_map: np.ndarray, value_map: Optional[np.ndarray] = None,
           valid_map: Optional[np.ndarray] = None, cam_pose: Optional[np.ndarray] = None,
           center_mode: CenterMode = CenterMode.none, merge: bool = True, keep_pose: bool = False,
           **kwargs: Dict[str, Any]) -> TopdownMap:
    """Plot the frame's local map and (by default) merge it into the world map
    (maps.py:2357-2406).  Returns the local map."""
    if self._native and merge and not keep_pose and valid_map is None:
      done = self._native_step(depth_map, value_map, cam_pose, center_mode, kwargs)
      if done is not None:
        return done
    topdown_map = self.plot(depth_map=depth_map, value_map=value_map, valid_map=valid_map, cam_pose=cam_pose,
                            center_mode=center_mode, **kwargs)
    if merge:
      self.merge(topdown_map, keep_pose=keep_pose)
    return topdown_map

  def plot(self, depth_map: np.ndarray, value_map: Optional[np.ndarray] = None,
           valid_map: Optional[np.ndarray] = None, cam_pose: Optional[np.ndarray] = None,
           center_mode: CenterMode = CenterMode.none, **kwargs: Dict[str, Any]) -> TopdownMap:
    """orth_project with get_height_map=True, wrapped as a TopdownMap that remembers the pose and
    offsets it was plotted with (maps.py:2408-2469)."""
    cam_pose = get(cam_pose, self.proj.cam_pose, np.array([0., 0., 0.], dtype=np.float32))
    width_offset, height_offset = self._compute_offsets(cam_pose=cam_pose, center_mode=center_mode, **kwargs)
    kwargs['width_offset'] = width_offset
    kwargs['height_offset'] = height_offset
    kwargs.pop('get_height_map', None)
    topdown_map, mask, height_map = self.proj.orth_project(
      depth_map=depth_map, value_map=value_map, valid_map=valid_map, cam_pose=cam_pose,
      get_height_map=True, **kwargs)
    clone_kwargs = {k: v for k, v in kwargs.items() if k in _CTOR_ARGS}
    return TopdownMap(topdown_map=topdown_map, mask=mask, height_map=height_map,
                      map_projector=self.proj.clone(cam_pose=cam_pose, **clone_kwargs),
                      is_height_map=(value_map is None and kwargs.get('label_map') is None))

  def merge(self, topdown_map: TopdownMap, keep_pose: bool = False, fill_value: Optional[float] = None,
            reduction: Optional[Reduction] = None) -> TopdownMap:
    """Fuse `topdown_map` into the world map, in the new map's camera frame unless `keep_pose`
    (maps.py:2471-2508)."""
    if self._world_map is None:
      self._world_map = TopdownMap(map_projector=self.proj.clone())
    old = self._world_map
    cam_pose = old.proj.cam_pose if keep_pose else topdown_map.proj.cam_pose
    if self._fixed is not None:
      self._world_map = merge_into_canvas(old, topdown_map, canvas_shape=self._fixed,
                                          map_projector=self.proj.clone(cam_pose=cam_pose),
                                          fill_value=fill_value, reduction=reduction)
    else:
      self._world_map = fuse_topdown_maps(old, topdown_map, map_projector=self.proj.clone(cam_pose=cam_pose),
                                          fill_value=fill_value, reduction=reduction)
    # both merges return either canvases they allocated, or the tensors of one of the two maps they were given
    mask = self._world_map.mask
    fresh = mask is not None and mask is not topdown_map.mask and mask is not old.mask
    self._owned = mask if fresh or (mask is old.mask and mask is self._owned) else None
    return self._world_map

  # ---- the step with its host side in C (csrc/dm_builder.cu) ----------------------------------------------------

  _NATIVE_KW = frozenset(("to_global", "width_offset", "height_offset", "map_width", "map_height", "label_map",
                          "num_classes"))
  _MAX_HANDLES = 4  # a value-map handle owns a projection workspace of C planes: keep the few recently used ones

  def _native_handle(self, key: tuple, dev: torch.device) -> "_NativeBuilder":
    """The handle of `key`, created on first use; the least recently used one beyond _MAX_HANDLES is destroyed."""
    nb = self._handles.pop(key, None)
    if nb is None:
      nb = _NativeBuilder(self.proj, key, dev)
    self._handles[key] = nb
    while len(self._handles) > self._MAX_HANDLES:
      self._handles.pop(next(iter(self._handles))).close()
    return nb

  @staticmethod
  def _native_values(depth_map, value_map, kwargs):
    """(kind, C, values, labels) of a step the C step can take, or None: kind "height" (C = 0), "values" (a CUDA
    float32 contiguous (b, C, H, W) value_map) or "labels" (a CUDA integer (b, 1, H, W) label_map, 1..63 classes).
    Argument errors are left to the general path, which reports them."""
    label_map, num_classes = kwargs.get("label_map"), kwargs.get("num_classes")
    b, _, H, W = depth_map.shape
    if label_map is not None:
      if (value_map is not None or num_classes is None or not torch.is_tensor(label_map) or not label_map.is_cuda
          or label_map.device != depth_map.device or label_map.dtype.is_floating_point or label_map.dtype is torch.bool
          or tuple(label_map.shape) != (b, 1, H, W) or not 1 <= int(num_classes) <= 63):
        return None
      C = int(num_classes)
      return "labels", C, None, _label_ids(label_map, C, depth_map.device)
    if num_classes is not None:
      return None
    if value_map is None:
      return "height", 0, None, None
    if (not torch.is_tensor(value_map) or value_map.device != depth_map.device or value_map.dtype is not torch.float32
        or value_map.dim() != 4 or value_map.shape[0] != b or value_map.shape[1] < 1
        or tuple(value_map.shape[2:]) != (H, W) or not value_map.is_contiguous()):
      return None
    return "values", int(value_map.shape[1]), value_map, None

  def _native_step(self, depth_map, value_map, cam_pose, center_mode, kwargs) -> Optional[TopdownMap]:
    """MapBuilder.step for the case dm_builder_* covers; None when the call needs the general path.  One sequence for
    height maps (C = 0: one plane) and value maps (C planes, their heights as C planes of the world map and one plane
    of the local map)."""
    proj = self.proj
    if (CenterMode(center_mode) is not CenterMode.none or not set(kwargs) <= self._NATIVE_KW or not proj.to_global
        or not torch.is_tensor(depth_map) or not depth_map.is_cuda or depth_map.dtype is not torch.float32
        or depth_map.dim() != 4 or depth_map.shape[1] != 1 or not depth_map.is_contiguous()):
      return None
    picked = self._native_values(depth_map, value_map, kwargs)
    if picked is None:
      return None
    kind, C, values, labels = picked
    kwargs = {k: v for k, v in kwargs.items() if k not in ("label_map", "num_classes")}
    get_kw = lambda name: get(kwargs.get(name), getattr(proj, name))
    scalars = [proj.cam_pitch, proj.cam_height, proj.map_res, get_kw("width_offset"), get_kw("height_offset"),
               get_kw("map_width"), get_kw("map_height")]
    if any(v is None or torch.is_tensor(v) or isinstance(v, (np.ndarray, list, tuple)) for v in scalars):
      return None
    try:
      red = utils._reduction_code(proj.reduction)
    except NotImplementedError:
      return None
    dev = depth_map.device
    b, _, H, W = depth_map.shape
    if (H, W) != (int(proj.height), int(proj.width)):
      return None
    world = self._world_map
    have_world = world is not None and not world.is_empty
    if have_world and not self._native_world_ok(world, b, dev, C):
      return None
    cam_pose = get(cam_pose, proj.cam_pose, np.array([0., 0., 0.], dtype=np.float32))
    plot_global = bool(get_kw("to_global"))
    woff, hoff = float(scalars[3]), float(scalars[4])
    Mw, Mh = int(scalars[5]), int(scalars[6])
    fill = proj.fill_value
    key = (b, H, W, dev.index, plot_global, woff, hoff, Mw, Mh, float(proj.cam_pitch), float(proj.cam_height),
           float(proj.map_res), proj.hfov, proj.vfov, proj.trunc_depth_min, proj.trunc_depth_max,
           proj.trunc_height_max, proj.clip_border, bool(proj.flip_h), fill, red, kind, C)
    nb = self._native_handle(key, dev)
    n = max(C, 1)   # planes per environment
    pose = prm.per_sample(cam_pose, b, (3,), "cam_pose").contiguous()
    # utils.py:325-326 with the reference's own torch-CPU ops (the last ulp of sin / cos matters)
    sin, cos = prm.yaw_sin_cos(pose)
    local = (torch.empty((b, n, Mh, Mw), dtype=torch.float32, device=dev),
             torch.empty((b, n, Mh, Mw), dtype=torch.bool, device=dev))
    if C:
      local += (torch.empty((b, 1, Mh, Mw), dtype=torch.float32, device=dev),)   # one height plane for all C channels
    inputs = nb.inputs(depth_map, values, labels, pose, sin, cos, local)
    stream = nat.stream_ptr(dev)
    def make_local():
      """The local map as plot() describes it (maps.py:2459-2469); offsets as compute_center_offsets returns them, and
      a value map's height map is the stride-0 expand orth_project returns.
      Built AFTER the step's kernels are queued: host bookkeeping belongs behind GPU work, not in front of it."""
      local_kw = {k: v for k, v in kwargs.items() if k in _CTOR_ARGS}
      local_kw["width_offset"] = torch.tensor([woff], dtype=torch.float32)
      local_kw["height_offset"] = torch.tensor([hoff], dtype=torch.float32)
      top, mask = local[:2]
      height = torch.broadcast_to(local[2], top.shape) if C else top
      return TopdownMap(topdown_map=top, mask=mask, height_map=height,
                        map_projector=proj.clone(cam_pose=cam_pose, **local_kw), is_height_map=C == 0)
    def world_map(canvases, map_projector):
      return TopdownMap(topdown_map=canvases[0], mask=canvases[1], height_map=canvases[2] if C else canvases[0],
                        map_projector=map_projector, is_height_map=C == 0)
    target = proj.clone(cam_pose=cam_pose)
    with torch.cuda.device(dev):
      if self._fixed is not None:
        Hc, Wc = self._fixed
        if have_world:
          canvases = nb.canvases(world)
        else:
          canvases = [torch.empty((b, n, Hc, Wc), dtype=dt, device=dev) for dt in nb.dtypes]
          top, mask, height = canvases[0], canvases[1], canvases[2] if C else None
          nat.check(nat.lib().dm_fuse_canvas_init_f32(top.data_ptr(), mask.data_ptr(), nat.ptr(height), top.numel(),
                                                      nb.fill, stream), "dm_fuse_canvas_init_f32")
          self._owned = canvases[1]
        nb.step_fixed(inputs, nb.map_ref(canvases, Hc, Wc, Wc / 2., Hc / 2.), stream)
        self._world_map = world_map(canvases, target.clone(to_global=True, width_offset=Wc / 2., height_offset=Hc / 2.,
                                                           map_width=Wc, map_height=Hc))
        return make_local()
      wref = None
      if have_world:
        box = world._tracked_box.box if _tracked_box_valid(world, target, dev) else None
        wref = nb.map_ref(nb.canvases(world), world.mask.shape[-2], world.mask.shape[-1],
                          float(world.proj.width_offset), float(world.proj.height_offset), box,
                          _tracked_planes(world, dev, b * n))
      # Everything the merge needs that does not depend on the bounding box is set up BEFORE the call that waits for it:
      # the GPU idles from the moment the box arrives until the merge kernels are queued.  The new canvas is as a rule
      # in the size class of the old one (the map grows by a few cells per step), so canvases of that class are taken
      # from the allocator ahead of the sync and only replaced when the box asks for more.
      track = nb.fill == nb.fill
      next_box = torch.empty((5,), dtype=torch.int64, device=dev) if track else None
      next_planes = torch.empty((b * n, 4), dtype=torch.int32, device=dev) if track else None
      spec = None
      if have_world and world.mask.numel() >= (1 << 18):
        cap = _canvas_cap(world.mask.numel())
        spec = [torch.empty((cap,), dtype=dt, device=dev) for dt in nb.dtypes]
      # ... and their fill is queued behind the box's copy: it runs while the host waits for the box
      # (prefilled: the old map's cells + 2 % — the map grows by a row or a column now and then; the merge fills
      # whatever tail the new map has beyond that, and the rest of the size class stays untouched)
      n_guess = 0 if spec is None else min(spec[0].numel(), world.mask.numel() + world.mask.numel() // 50 + 4096)
      nb.plot(inputs, wref, spec, n_guess, stream)
      local_map = make_local()  # while the projection, the box reduction and the prefill run
      shape = nb.wait()
      if shape.n_valid == 0:  # maps.py:2217-2225
        self._world_map = TopdownMap(topdown_map=local_map.topdown_map, mask=local_map.mask,
                                     height_map=local_map.height_map, map_projector=target)
        self._owned = None
        return local_map
      mh, mw = shape.map_height, shape.map_width
      n_new = b * n * mh * mw
      if spec is not None and (1 << 18) <= n_new <= spec[0].numel():
        canvases = [t[:n_new].view(b, n, mh, mw) for t in spec]
      else:
        # the map outgrew the guess: the speculative canvases go back to the allocator BEFORE the new ones are taken,
        # so that canvases of the old class are not held next to the old map and the new one
        # (the prefill queued on them is ordered before any later use of their blocks on this stream)
        spec = None
        canvases = [_alloc_canvas((b, n, mh, mw), dt, dev) for dt in nb.dtypes]
      nb.merge(nb.map_ref(canvases, mh, mw, shape.width_offset, shape.height_offset, next_box, next_planes), stream)
    new_proj = target.clone(width_offset=torch.tensor([shape.width_offset], dtype=torch.float32),
                            height_offset=torch.tensor([shape.height_offset], dtype=torch.float32),
                            map_width=mw, map_height=mh)
    merged = world_map(canvases, new_proj)
    if track:
      merged._tracked_box = _TrackedBox(next_box, merged.mask, new_proj, next_planes)
    # (the scatter pass still reads the old world map and the local map on the stream: torch's caching allocator
    # hands freed blocks to later work of the same stream only, so dropping the old map here is safe)
    self._world_map, self._owned = merged, merged.mask
    return local_map

  def _native_world_ok(self, world: TopdownMap, b: int, dev: torch.device, C: int = 0) -> bool:
    """The world map is one the C step can take as it is: a contiguous (b, 1, h, w) float32 height map + bool mask
    (C = 0), or a contiguous (b, C, h, w) float32 value map with (b, C, h, w) height planes + bool mask (C >= 1), on
    `dev`, in the global frame, with this builder's resolution / flip and scalar offsets."""
    p, proj = world.proj, self.proj
    top, mask = world.topdown_map, world.mask
    if not (bool(world.is_height_map) == (C == 0) and p is not None and p.to_global and torch.is_tensor(top)
            and torch.is_tensor(mask)):
      return False
    if self._fixed is not None and tuple(top.shape[-2:]) != self._fixed:
      return False
    ok_t = lambda t, dt: (t.device == dev and t.dtype is dt and t.dim() == 4 and t.shape[0] == b
                          and t.shape[1] == max(C, 1) and t.is_contiguous())
    if not (ok_t(top, torch.float32) and ok_t(mask, torch.bool) and top.shape == mask.shape):
      return False
    hm = world.height_map
    if C > 0 and not (torch.is_tensor(hm) and ok_t(hm, torch.float32) and hm.shape == top.shape):
      return False
    def one(v):
      if v is None:
        return False
      if torch.is_tensor(v):
        return v.numel() == 1
      return np.asarray(v).size == 1
    return (float(p.map_res) == float(proj.map_res) and bool(p.flip_h) == bool(proj.flip_h)
            and one(p.width_offset) and one(p.height_offset))

  def _compute_offsets(self, cam_pose: np.ndarray, width_offset: Optional[np.ndarray] = None,
                       height_offset: Optional[np.ndarray] = None, map_res: Optional[float] = None,
                       map_width: Optional[int] = None, map_height: Optional[int] = None,
                       to_global: Optional[bool] = None, center_mode: Optional[CenterMode] = None,
                       **kw_) -> Tuple[torch.Tensor, torch.Tensor]:
    return self.proj.compute_center_offsets(cam_pose=cam_pose, width_offset=width_offset,
                                            height_offset=height_offset, map_res=map_res, map_width=map_width,
                                            map_height=map_height, to_global=to_global, center_mode=center_mode)
