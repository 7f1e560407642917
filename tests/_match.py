"""score_poses as its definition composes it: for each candidate pose, TopdownMap.select_egocentric's composition of the
oracle's public-function restatements (tests/_egocentric.crop_egocentric) applied to the planes, ANDed with the window
and counted; and the case generators the tests share."""
import numpy as np

from tests._egocentric import crop_egocentric


def score_poses(planes, window, src_woff, src_hoff, map_res, flip_h, cam_poses, woff, hoff):
  """planes bool (b, C, Hs, Ws); window bool (b, 1 or C, h, w); cam_poses (n, 3) or (b, n, 3); offsets 1 or b values.
  Returns int32 (b, C, n)."""
  planes = np.asarray(planes, dtype=bool)
  window = np.asarray(window, dtype=bool)
  b, C = planes.shape[:2]
  h, w = window.shape[-2:]
  poses = np.asarray(cam_poses, dtype=np.float32)
  poses = np.broadcast_to(poses.reshape(-1, poses.shape[-2], 3), (b, poses.shape[-2], 3))
  top = planes.astype(np.float32)
  out = np.empty((b, C, poses.shape[1]), dtype=np.int32)
  for k in range(poses.shape[1]):
    _, mask, _ = crop_egocentric(top, planes, None, src_woff, src_hoff, map_res, flip_h,
                                 np.ascontiguousarray(poses[:, k]), w, h, woff, hoff, 0.)
    out[:, :, k] = (mask & window).sum(axis=(2, 3))
  return out


def random_planes(rng, shape, density):
  """Bool planes, True with probability `density` (0 and 1 give all-False and all-True)."""
  return rng.random(shape) < density


def lattice(center, steps, res_xz, res_yaw):
  """(n, 3) float32 candidates: center + (i dx, j dz, k dyaw) for i, j, k in -steps..steps, yaw fastest."""
  r = np.arange(-steps, steps + 1)
  i, j, k = np.meshgrid(r, r, r, indexing="ij")
  d = np.stack((i.ravel() * res_xz, j.ravel() * res_xz, k.ravel() * res_yaw), axis=1)
  return (np.asarray(center, np.float32)[..., None, :] + d.astype(np.float32)).astype(np.float32)
