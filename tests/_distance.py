"""The definition of distance_transform, restated without the library: scipy.ndimage.distance_transform_edt per plane
cast to float32 (inf on planes without a False cell), a check of `nearest` that holds for any tie choice, and a brute-force oracle.
The mask generators are tests/_components.py's `pattern`."""
import numpy as np
from scipy import ndimage


def oracle(mask: np.ndarray) -> np.ndarray:
  """(..., H, W) bool -> float32 distances: scipy per plane; +inf on every cell of a plane without a False cell."""
  H, W = mask.shape[-2:]
  planes = mask.reshape(-1, H, W)
  out = np.empty(planes.shape, np.float32)
  for i, p in enumerate(planes):
    out[i] = ndimage.distance_transform_edt(p).astype(np.float32) if not p.all() else np.inf
  return out.reshape(mask.shape)


def check_nearest(mask: np.ndarray, dist: np.ndarray, nearest: np.ndarray) -> None:
  """nearest (..., H, W, 2) [x, z] against mask and dist, whatever the tie choice: in range, False in the mask, at
  exactly the squared distance dist was rounded from, and the cell itself on False cells; -1 on planes without a False
  cell."""
  H, W = mask.shape[-2:]
  m = mask.reshape(-1, H, W)
  d = dist.reshape(-1, H, W)
  n = nearest.reshape(-1, H, W, 2)
  assert nearest.shape == mask.shape + (2,) and nearest.dtype == np.int32
  r, c = np.indices((H, W))
  for p in range(m.shape[0]):
    x, z = n[p, ..., 0], n[p, ..., 1]
    if m[p].all():
      assert (x == -1).all() and (z == -1).all(), f"plane {p}: no False cell, so nearest must be -1"
      continue
    assert ((x >= 0) & (x < W) & (z >= 0) & (z < H)).all(), f"plane {p}: nearest out of range"
    assert not m[p][z, x].any(), f"plane {p}: nearest is a True cell"
    d2 = (r - z).astype(np.int64) ** 2 + (c - x).astype(np.int64) ** 2
    assert np.array_equal(np.sqrt(d2.astype(np.float64)).astype(np.float32), d[p]), \
        f"plane {p}: nearest is not at the returned distance"
    assert (x[~m[p]] == c[~m[p]]).all() and (z[~m[p]] == r[~m[p]]).all(), f"plane {p}: a False cell is not its own"


def brute_force(plane: np.ndarray) -> np.ndarray:
  """(H, W) bool with a False cell -> float32 distances: the minimum over all False cells, in float64."""
  r, c = np.indices(plane.shape)
  fr, fc = np.nonzero(~plane)
  d2 = (r[..., None] - fr) ** 2 + (c[..., None] - fc) ** 2
  return np.sqrt(d2.min(-1).astype(np.float64)).astype(np.float32)


def scipy_nearest(plane: np.ndarray) -> np.ndarray:
  """scipy's return_indices (2, H, W) [row, column] as this library's (H, W, 2) [x, z]."""
  _, idx = ndimage.distance_transform_edt(plane, return_indices=True)
  return np.stack([idx[1], idx[0]], -1).astype(np.int32)


def sqrtf_plane() -> np.ndarray:
  """(8, 6000) bool, False only at (0, 0): squared distances up to 7^2 + 5999^2 > 2^24, and on 1198 cells
  np.sqrt(float32(d2)) differs from scipy's rounding (a 2 x 6000 plane has none: d2 = c^2 and c^2 + 1 round alike)."""
  plane = np.ones((8, 6000), bool)
  plane[0, 0] = False
  return plane
