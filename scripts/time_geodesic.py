#!/usr/bin/env python
"""geodesic_distance on config-4 world maps and on a spiral maze: one JSON line per case.

Cases:
  growing / fixed   the world maps of a 32-environment, 100-step MapBuilder walk over synth room scenes
                    (bench.BuilderWorkload geometry), on the growing world map and on 2400 x 2400 fixed canvases;
                    traversable = seen and not above 0.2 m ("seen"), or that or unseen ("unknown free"); the source is
                    each agent's cell (TopdownMap.geodesic_distance's default).
  spiral N          one N x N one-cell-corridor spiral maze (tests/_geodesic.py), source in its outer corner: about
                    N * N / 2 cells on one path, the worst case for the kernel's round count.
Arms:
  kernel   dm_geodesic_distance_i32: GPU ms per call from CUDA events around --calls calls (warm shapes), and the
           call time (host clock from the call to the end of a device synchronise, median).
  torch    shifted-neighbour min-plus relaxation on the GPU, iterated until unchanged, checked every 32 iterations.
  scipy    what users do now: a device-to-host copy and scipy.sparse.csgraph.dijkstra per environment.
The three must agree exactly (asserted on the environments each arm ran).  On the 2400 x 2400 canvases the torch arm
runs the first 4 environments and the scipy arm the first 2, and the torch arm skips spirals above 256 x 256 (each
iteration advances the front by one cell); every line says how many environments each arm ran.

usage: python scripts/time_geodesic.py [--calls 10] [--out results/geodesic.jsonl]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from scipy.sparse import csr_matrix  # noqa: E402
from scipy.sparse.csgraph import dijkstra  # noqa: E402

import dungeon_maps_b200 as dmap  # noqa: E402
from scripts.time_egocentric import EPISODE, Walk  # noqa: E402
from scripts.time_reset_envs import card, make_builder  # noqa: E402
from tests._geodesic import STEPS, spiral_maze  # noqa: E402

L2_BYTES = 126 * 2 ** 20


def torch_baseline(trav, src, check_every=32):
  """(b, H, W) bool -> int32 distances: min-plus relaxation over the 8 shifted neighbours until nothing changes."""
  inf = 1 << 30
  b, H, W = trav.shape
  tp = F.pad(trav, (1, 1, 1, 1))
  oks = []
  for dr, dc, _ in STEPS:
    ok = trav.clone()
    if dr and dc:
      ok &= tp[:, 1 - dr:1 - dr + H, 1:1 + W] & tp[:, 1:1 + H, 1 - dc:1 - dc + W]
    oks.append(ok)
  d = torch.where(src, 0, inf).to(torch.int32)
  iters = 0
  while True:
    prev = d
    for _ in range(check_every):
      p = F.pad(d, (1, 1, 1, 1), value=inf)
      best = d
      for (dr, dc, w), ok in zip(STEPS, oks):
        best = torch.minimum(best, torch.where(ok, p[:, 1 - dr:1 - dr + H, 1 - dc:1 - dc + W] + w, inf))
      d = best
    iters += check_every
    if torch.equal(d, prev):
      return torch.where(d >= inf, -1, d), iters


def scipy_dijkstra(trav, src):
  """(H, W) bool numpy grids -> int32 distances with scipy's Dijkstra over the same graph."""
  H, W = trav.shape
  ids = np.arange(H * W, dtype=np.int64).reshape(H, W)
  tp = np.pad(trav, 1)
  rows, cols, costs = [], [], []
  for dr, dc, w in STEPS:     # edges u -> v = u + (dr, dc), listed per destination v
    ok = trav.copy()
    valid = np.zeros((H, W), bool)
    valid[max(dr, 0):H + min(dr, 0), max(dc, 0):W + min(dc, 0)] = True   # u = v - (dr, dc) inside the grid
    ok &= valid
    if dr and dc:
      ok &= tp[1 - dr:1 - dr + H, 1:1 + W] & tp[1:1 + H, 1 - dc:1 - dc + W]
    v = ids[ok]
    rows.append(v - dr * W - dc)
    cols.append(v)
    costs.append(np.full(v.shape, w, np.float32))
  g = csr_matrix((np.concatenate(costs), (np.concatenate(rows), np.concatenate(cols))), shape=(H * W, H * W))
  starts = np.flatnonzero(src)
  if len(starts) == 0:
    return np.full((H, W), -1, np.int32)
  d = dijkstra(g, directed=True, indices=starts, min_only=True)
  return np.where(np.isinf(d), -1, d).astype(np.int32).reshape(H, W)


def time_case(name, trav, src, args, torch_envs, scipy_envs, extra):
  b, H, W = trav.shape
  out = dmap.geodesic_distance(trav, src)          # warm the shape
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(args.calls):
    out = dmap.geodesic_distance(trav, src)
  e1.record()
  torch.cuda.synchronize()
  kernel_ms = e0.elapsed_time(e1) / args.calls
  calls = []
  for _ in range(args.calls):
    t0 = time.perf_counter()
    dmap.geodesic_distance(trav, src)
    torch.cuda.synchronize()
    calls.append((time.perf_counter() - t0) * 1e3)
  from dungeon_maps_b200 import _native as nat
  nat.device_status()
  line = dict(card(), case=name, b=b, H=H, W=W, traversable_cells=int(trav.sum()),
              input_output_bytes=b * H * W * 6, larger_than_l2=b * H * W * 6 > L2_BYTES,
              kernel_ms=round(kernel_ms, 4), call_ms_median=round(float(np.median(calls)), 4), **extra)
  mask = src if src.dtype is torch.bool else None
  if mask is None:
    mask = torch.zeros_like(trav)
    c = src.to(trav.device)
    mask[torch.arange(b, device=trav.device), c[:, 1], c[:, 0]] = True
  if torch_envs:
    k = min(torch_envs, b)
    tb, tm = trav[:k].contiguous(), mask[:k].contiguous()
    torch_baseline(tb, tm, 32)                       # warm
    torch.cuda.synchronize()
    e0.record()
    want, iters = torch_baseline(tb, tm)
    e1.record()
    torch.cuda.synchronize()
    assert torch.equal(want, out[:k]), f"{name}: the torch baseline differs"
    line.update(torch_envs=k, torch_ms=round(e0.elapsed_time(e1), 3), torch_iterations=iters)
  else:
    line.update(torch_envs=0, torch_ms="not measured")
  if scipy_envs:
    k = min(scipy_envs, b)
    t0 = time.perf_counter()
    th, mh = trav[:k].cpu().numpy(), mask[:k].cpu().numpy()
    got = np.stack([scipy_dijkstra(th[i], mh[i]) for i in range(k)])
    scipy_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(got, out[:k].cpu().numpy()), f"{name}: scipy differs"
    line.update(scipy_envs=k, scipy_ms=round(scipy_ms, 1), scipy_ms_per_env=round(scipy_ms / k, 1))
  else:
    line.update(scipy_envs=0, scipy_ms="not measured")
  print(json.dumps(line), flush=True)
  return line


def world_maps(fixed, dev):
  walk = Walk(32, 0, dev)
  builder = make_builder(dev)
  if fixed:
    builder = dmap.MapBuilder(map_projector=builder.proj, fixed_canvas=(2400, 2400))
  for t in range(EPISODE):
    walk.step(builder, t)
  torch.cuda.synchronize()
  return builder.world_map


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--calls", type=int, default=10)
  ap.add_argument("--out", default=None)
  ap.add_argument("--cases", default="growing,fixed,spiral256,spiral1024")
  args = ap.parse_args()
  dev = torch.device("cuda", 0)
  lines = []
  for case in args.cases.split(","):
    if case in ("growing", "fixed"):
      world = world_maps(case == "fixed", dev)
      hm, seen = world.height_map[:, 0], world.mask[:, 0]
      cam = world.get_camera()
      for variant in ("seen", "unknown free"):
        free = seen & (hm <= 0.2)
        if variant == "unknown free":
          free = free | ~seen
        big = case == "fixed"
        lines.append(time_case(f"{case} world map, {variant}", free.contiguous(), cam, args,
                               torch_envs=4 if big else 32, scipy_envs=2 if big else 32,
                               extra=dict(source="agent cell", steps=EPISODE)))
    elif case.startswith("spiral"):
      n = int(case[len("spiral"):])
      trav = torch.from_numpy(spiral_maze(n, n))[None].to(dev)
      src = torch.zeros_like(trav)
      src[0, 0, 0] = True
      lines.append(time_case(f"spiral {n}", trav, src, args, torch_envs=1 if n <= 256 else 0, scipy_envs=1,
                             extra=dict(source="outer corner")))
  if args.out:
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
      for line in lines:
        f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
  main()
