"""The definition of connected_components, restated without the library: scipy.ndimage.label per plane with the two
structures, np.bincount for the sizes, and mask generators (spiral mazes, checkerboards, stripes, rooms)."""
import numpy as np
from scipy import ndimage

from tests._geodesic import spiral_maze

STRUCTURES = {4: ndimage.generate_binary_structure(2, 1), 8: np.ones((3, 3), bool)}
# site-percolation thresholds of the square lattice: the densities where components are largest and most winding
PERCOLATION = {4: 0.593, 8: 0.407}


def label_plane(plane: np.ndarray, connectivity: int):
  """(H, W) bool -> (labels int32, K, sizes int32)."""
  labels, k = ndimage.label(plane, STRUCTURES[connectivity])
  labels = labels.astype(np.int32)
  per = np.bincount(labels.ravel(), minlength=k + 1).astype(np.int32)
  per[0] = 0
  return labels, int(k), per[labels]


def oracle(mask: np.ndarray, connectivity: int):
  """(..., H, W) bool -> labels (..., H, W) int32, counts (...) int32, sizes (..., H, W) int32."""
  H, W = mask.shape[-2:]
  planes = mask.reshape(-1, H, W)
  out = [label_plane(p, connectivity) for p in planes]
  labels = np.stack([o[0] for o in out]).reshape(mask.shape)
  counts = np.array([o[1] for o in out], np.int32).reshape(mask.shape[:-2])
  sizes = np.stack([o[2] for o in out]).reshape(mask.shape)
  return labels, counts, sizes


def checkerboard(H: int, W: int) -> np.ndarray:
  """(H, W) bool with (0, 0) set: one component under 8-connectivity, ceil(H * W / 2) under 4-connectivity."""
  r, c = np.indices((H, W))
  return (r + c) % 2 == 0


def stripes(H: int, W: int, vertical: bool) -> np.ndarray:
  """One-cell stripes one cell apart: columns (vertical) or rows."""
  r, c = np.indices((H, W))
  return (c if vertical else r) % 2 == 0


def rooms(H: int, W: int) -> np.ndarray:
  """Free space of rooms: walls every 37 rows / 29 columns with doors, as in the geodesic tests."""
  t = np.ones((H, W), bool)
  t[36::37, :] = False
  t[:, 28::29] = False
  t[36::37, 5::29] = True
  t[10::37, 28::29] = True
  return t


def pattern(kind: str, H: int, W: int, rng, connectivity: int = 8) -> np.ndarray:
  if kind.startswith("random"):
    density = PERCOLATION[connectivity] if kind == "random percolation" else float(kind.split()[1])
    return rng.random((H, W)) < density
  if kind == "spiral":
    return spiral_maze(H, W)
  if kind == "checkerboard":
    return checkerboard(H, W)
  if kind == "vertical stripes":
    return stripes(H, W, True)
  if kind == "horizontal stripes":
    return stripes(H, W, False)
  if kind == "rooms":
    return rooms(H, W)
  if kind == "all true":
    return np.ones((H, W), bool)
  if kind == "all false":
    return np.zeros((H, W), bool)
  raise ValueError(kind)
