"""TopdownMap.select_egocentric as its definition composes it from the oracle's public-function restatements
(oracle/dm_oracle.py): map_dequantize of the window's cells, local_to_global_space with the pose (crop_h * crop_w points
per sample, which picks the fused or naive rotation as the reference's bmm does), map_quantize with the source's
offsets, and a numpy gather with the merge's fills outside the source."""
import numpy as np

from oracle import dm_oracle as orc


def window_cells(b, crop_w, crop_h):
  """(b, crop_h * crop_w) float32 column and row indices of every window cell, row-major."""
  r, c = np.divmod(np.arange(crop_h * crop_w), crop_w)
  return (np.ascontiguousarray(np.broadcast_to(c, (b, c.size)), dtype=np.float32),
          np.ascontiguousarray(np.broadcast_to(r, (b, r.size)), dtype=np.float32))


def _rows(x, b, tail=()):
  a = np.asarray(x, dtype=np.float32).reshape((-1,) + tail)
  return np.ascontiguousarray(np.broadcast_to(a, (b,) + tail)) if a.shape[0] == 1 else a


def crop_egocentric(topdown, mask, height, src_woff, src_hoff, map_res, flip_h, pose, crop_w, crop_h, woff, hoff,
                    fill_value):
  """topdown / mask (b, C, Hs, Ws), height (b, C or 1, Hs, Ws) or None (a height map); pose (1 or b, 3); offsets 1 or b
  values.  Returns (topdown, mask, height) windows; height None for a height map."""
  topdown = np.asarray(topdown, dtype=np.float32)
  b, C, Hs, Ws = topdown.shape
  n = crop_h * crop_w
  xb, zb = window_cells(b, crop_w, crop_h)
  lx, lz = orc.map_dequantize(xb, zb, _rows(woff, b), _rows(hoff, b), map_res, crop_h, flip_h)
  pts = np.ascontiguousarray(np.stack((lx, np.zeros_like(lx), lz), axis=-1))
  g = orc.transform_points(pts, [orc.to_global_steps(_rows(pose, b, (3,)), n)])
  X, Z = orc.map_quantize(g[..., 0], g[..., 2], _rows(src_woff, b), _rows(src_hoff, b), map_res, Hs, flip_h)
  inside = (X >= 0) & (X < Ws) & (Z >= 0) & (Z < Hs)
  cell = np.where(inside, Z * Ws + X, 0)

  def gather(planes, fill):
    p = np.asarray(planes).reshape(b, planes.shape[1], Hs * Ws)
    got = np.take_along_axis(p, np.broadcast_to(cell[:, None, :], (b, p.shape[1], n)), axis=2)
    return np.where(inside[:, None, :], got, np.asarray(fill, dtype=p.dtype)).reshape(b, p.shape[1], crop_h, crop_w)

  out_h = None if height is None else gather(np.asarray(height, dtype=np.float32), -np.inf)
  return gather(topdown, fill_value), gather(np.asarray(mask, dtype=bool), False), out_h
