#!/usr/bin/env python
"""TopdownMap.select_egocentric at BASELINE config-4 geometry (480x640 depth -> 400x400 local maps at 3 cm, the
bench.BuilderWorkload walk), 256x256 windows: one JSON line per case and arm.

Cases: 32 environments with height maps on the growing world map and on 2400x2400 fixed canvases, and 8 environments
with 16 classes given as class ids (label_map=, num_classes=) on the growing world map.  Each case first runs the
100-step walk, then times windows of that world map at the walk's 100 poses in turn (the 10-75 MB of output per call
fit the 126 MB L2; the world maps do not).  Arms, alternated in one process:
  A  select_egocentric (dm_crop_egocentric_f32);
  B  the same window composed from the public functions: map_dequantize -> local_to_global_space -> map_quantize ->
     torch gather (bit-identical to A, asserted);
  C  a hand-written affine_grid + grid_sample(mode='nearest', align_corners=True) of the value planes (and the heights
     of value maps; no mask): for speed only, it is NOT bit-identical (other rounding, zeros instead of the fill).
Per arm: GPU ms per call from CUDA events around the loop and host ms per call (the enqueue).  For A also: the
kernel's device time per call from a torch.profiler pass, the bytes it moves (output bytes + one gathered read per
output element, from shapes), and the rate of a device copy of the same byte count timed in the same run.  Last, the
config-4 step time with and without one window per step.

usage: python scripts/time_egocentric.py [--calls 200] [--repeat 2] [--cases all]
"""
import argparse
import json
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import bench  # noqa: E402
import dungeon_maps_b200 as dmap  # noqa: E402
from dungeon_maps_b200 import synth  # noqa: E402
from scripts.time_reset_envs import card, make_builder  # noqa: E402

EPISODE = 100
CROP = 256


class Walk:
  def __init__(self, B, C, dev):
    self.B, self.C = B, C
    w = bench.BuilderWorkload(argparse.Namespace(scene="room"))
    w.B = B
    self.poses = w.walk(B, EPISODE, 0)
    self.depth = w.frames_for(self.poses, dev, 0)
    self.labels = None
    if C:
      pool = [synth.block_labels(B, C, 480, 640, seed=t, device=dev).to(torch.uint8) for t in range(16)]
      self.labels = [pool[t % 16] for t in range(EPISODE)]
    self.kw = dict(to_global=False, width_offset=bench.MW / 2., height_offset=0., map_width=bench.MW,
                   map_height=bench.MH)

  def step(self, builder, t):
    kw = self.kw if not self.C else dict(self.kw, label_map=self.labels[t % EPISODE], num_classes=self.C)
    builder.step(self.depth[t % EPISODE], cam_pose=self.poses[t % EPISODE], **kw)


def composed(world, pose):
  """Arm B: the definition with the public functions."""
  top = world.topdown_map
  b, C, Hs, Ws = top.shape
  p = world.proj
  n = CROP * CROP
  idx = torch.arange(n, device=top.device)
  xb = (idx % CROP).to(torch.float32).expand(b, n)
  zb = (idx // CROP).to(torch.float32).expand(b, n)
  lx, lz = dmap.map_dequantize(xb, zb, CROP / 2., CROP / 2., p.map_res, CROP, p.flip_h)
  g = dmap.local_to_global_space(torch.stack((lx, torch.zeros_like(lx), lz), dim=-1), pose)
  X, Z = dmap.map_quantize(g[..., 0], g[..., 2], p.width_offset, p.height_offset, p.map_res, Hs, p.flip_h)
  inside = (X >= 0) & (X < Ws) & (Z >= 0) & (Z < Hs)
  cell = torch.where(inside, Z * Ws + X, torch.zeros_like(X))[:, None, :].expand(b, C, n)
  fill = dmap.get(p.fill_value, dmap.NINF)
  out = [torch.where(inside[:, None], top.view(b, C, -1).gather(2, cell), fill).view(b, C, CROP, CROP),
         torch.where(inside[:, None], world.mask.view(b, C, -1).gather(2, cell), False).view(b, C, CROP, CROP)]
  if not world.is_height_map:
    out.append(torch.where(inside[:, None], world.height_map.reshape(b, C, -1).gather(2, cell), -math.inf)
               .view(b, C, CROP, CROP))
  return out


def grid_sampled(world, pose):
  """Arm C: the window's cell centres as an affine map of the output pixel, resampled by grid_sample."""
  top = world.topdown_map
  b, C, Hs, Ws = top.shape
  p = world.proj
  res, u, v = float(p.map_res), CROP / 2., CROP / 2.
  yaw = pose[:, 2].double()
  c, s = torch.cos(yaw), torch.sin(yaw)
  # (lx, lz) = ((col - u) res, (CROP - 1 - row - v) res); the yaw rotation of local_to_global_space:
  # (gx, gz) = (c lx - s lz + x, s lx + c lz + z)
  # X = gx / res + W, Z = Hs - 1 - (gz / res + H); then columns / rows of both grids normalised (align_corners)
  W, H = float(p.width_offset), float(p.height_offset)
  k = (CROP - 1) / 2.
  ax, az = (Ws - 1) / 2., (Hs - 1) / 2.
  # col = k (xn + 1), row = k (yn + 1)
  lx_x, lx_0 = k * res, (k - u) * res                  # lx = lx_x xn + lx_0
  lz_y, lz_0 = -k * res, (CROP - 1 - k - v) * res      # lz = lz_y yn + lz_0
  gx = [c * lx_x, -s * lz_y, c * lx_0 - s * lz_0 + pose[:, 0].double()]
  gz = [s * lx_x, c * lz_y, s * lx_0 + c * lz_0 + pose[:, 1].double()]
  X = [gx[0] / res / ax, gx[1] / res / ax, (gx[2] / res + W) / ax - 1]
  Z = [-gz[0] / res / az, -gz[1] / res / az, (Hs - 1 - (gz[2] / res + H)) / az - 1]
  theta = torch.stack((torch.stack(X, 1), torch.stack(Z, 1)), 1).float().to(top.device, non_blocking=True)
  grid = F.affine_grid(theta, (b, C, CROP, CROP), align_corners=True)
  out = [F.grid_sample(top, grid, mode="nearest", align_corners=True)]
  if not world.is_height_map:
    out.append(F.grid_sample(world.height_map, grid, mode="nearest", align_corners=True))
  return out


def timed(fn, calls, poses):
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  for i in range(3):
    fn(poses[i % EPISODE])
  torch.cuda.synchronize()
  h0 = time.perf_counter()
  e0.record()
  for i in range(calls):
    fn(poses[i % EPISODE])
  h1 = time.perf_counter()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / calls, (h1 - h0) * 1e3 / calls


def kernel_us(world, poses, calls):
  from torch.profiler import ProfilerActivity, profile
  copy_src = torch.empty(traffic_bytes(world) // 2, dtype=torch.uint8, device=world.mask.device)
  copy_dst = torch.empty_like(copy_src)
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for i in range(calls):
      world.select_egocentric(CROP, CROP, cam_pose=poses[i % EPISODE])
      copy_dst.copy_(copy_src)
    torch.cuda.synchronize()
  us = {"crop_egocentric": [0., 0], "copy": [0., 0]}
  for e in prof.events():
    if e.device_type != torch.autograd.DeviceType.CUDA:
      continue
    t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    key = "crop_egocentric" if "crop_egocentric" in e.name else "copy" if "DtoD" in e.name else None
    if key:
      us[key][0] += t
      us[key][1] += 1
  return {k: v[0] / max(v[1], 1) for k, v in us.items()}, us["crop_egocentric"][1]


def traffic_bytes(world):
  """Bytes the kernel moves, from shapes: every output element written once and its source element read once."""
  b, C = world.mask.shape[:2]
  per = 4 + 1 + (0 if world.is_height_map else 4)   # value, mask, height
  return 2 * b * C * CROP * CROP * per


def copy_rate(nbytes, dev, calls=50):
  a = torch.empty(nbytes // 2, dtype=torch.uint8, device=dev)
  o = torch.empty_like(a)
  o.copy_(a)
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(calls):
    o.copy_(a)
  e1.record()
  torch.cuda.synchronize()
  ms = e0.elapsed_time(e1) / calls
  return ms, nbytes / ms * 1e-6   # GB/s


def run_case(B, C, fixed, args, dev):
  walk = Walk(B, C, dev)
  bld = make_builder(dev)
  if fixed:
    bld = dmap.MapBuilder(map_projector=bld.proj, fixed_canvas=(2400, 2400))
  for t in range(EPISODE):
    walk.step(bld, t)
  torch.cuda.synchronize()
  world = bld.world_map
  poses = [walk.poses[t] for t in range(EPISODE)]
  case = {"envs": B, "classes": C or None, "maps": "class ids" if C else "height",
          "world": "fixed 2400x2400" if fixed else "growing", "world_shape": list(world.mask.shape),
          "window": [CROP, CROP]}
  a = world.select_egocentric(CROP, CROP, cam_pose=poses[7])
  bb = composed(world, poses[7])
  assert torch.equal(a.topdown_map.view(torch.int32), bb[0].view(torch.int32)) and torch.equal(a.mask, bb[1])
  if C:
    assert torch.equal(a.height_map.contiguous().view(torch.int32), bb[2].view(torch.int32))
  del a, bb
  arms = {"A": lambda p: world.select_egocentric(CROP, CROP, cam_pose=p),
          "B": lambda p: composed(world, p), "C": lambda p: grid_sampled(world, p)}
  nbytes = traffic_bytes(world)
  for rep in range(args.repeat):
    for name, fn in arms.items():
      ms, host = timed(fn, args.calls, poses)
      line = dict(case, arm=name, repeat=rep, calls=args.calls, gpu_ms_per_call=round(ms, 4),
                  host_ms_per_call=round(host, 4))
      if name == "A":
        line["bytes_per_call"] = nbytes
        line["GB_per_s_from_events"] = round(nbytes / ms * 1e-6, 1)
      if name == "C":
        line["note"] = "not bit-identical to A (grid_sample rounding, zero padding); value planes only, no mask"
      print(json.dumps(line), flush=True)
    copy_ms, copy_gbs = copy_rate(nbytes, dev)
    print(json.dumps(dict(case, arm="device copy of the same byte count", repeat=rep, ms=round(copy_ms, 4),
                          GB_per_s=round(copy_gbs, 1))), flush=True)
  kus, n = kernel_us(world, poses, args.profile_calls)
  print(json.dumps(dict(case, profile="torch.profiler, CUDA activities", calls=n,
                        kernel_us_per_call=round(kus["crop_egocentric"], 2),
                        kernel_GB_per_s=round(nbytes / kus["crop_egocentric"] * 1e-3, 1),
                        copy_us_same_bytes=round(kus["copy"], 2),
                        copy_GB_per_s=round(nbytes / max(kus["copy"], 1e-9) * 1e-3, 1))), flush=True)
  del world, bld
  # the config-4 loop with and without one window per step, alternated
  for rep in range(args.repeat):
    for with_window in (False, True):
      b2 = make_builder(dev)
      if fixed:
        b2 = dmap.MapBuilder(map_projector=b2.proj, fixed_canvas=(2400, 2400))
      for t in range(EPISODE):
        walk.step(b2, t)
      torch.cuda.synchronize()
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for t in range(EPISODE, EPISODE + args.steps):
        walk.step(b2, t)
        if with_window:
          b2.world_map.select_egocentric(CROP, CROP)
      e1.record()
      torch.cuda.synchronize()
      ms = e0.elapsed_time(e1) / args.steps
      print(json.dumps(dict(case, loop="config-4 step", with_window=with_window, repeat=rep, steps=args.steps,
                            ms_per_step=round(ms, 4), env_steps_per_s=round(B / ms * 1e3, 1))), flush=True)
      del b2
  del walk
  torch.cuda.empty_cache()


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--calls", type=int, default=200)
  ap.add_argument("--profile-calls", type=int, default=50)
  ap.add_argument("--steps", type=int, default=100, help="timed config-4 steps, after one episode of warm-up")
  ap.add_argument("--repeat", type=int, default=2)
  ap.add_argument("--cases", default="all", help="all | height | fixed | labels")
  args = ap.parse_args()
  if min(args.calls, args.profile_calls, args.steps, args.repeat) < 1:
    ap.error("--calls, --profile-calls, --steps and --repeat must be >= 1")
  if not torch.cuda.is_available():
    sys.exit("time_egocentric.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  print(json.dumps(card()), flush=True)
  cases = {"height": (32, 0, False), "fixed": (32, 0, True), "labels": (8, 16, False)}
  for name, (B, C, fixed) in cases.items():
    if args.cases in ("all", name):
      run_case(B, C, fixed, args, dev)


if __name__ == "__main__":
  np.set_printoptions(precision=4)
  main()
