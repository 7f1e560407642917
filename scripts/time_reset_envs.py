#!/usr/bin/env python
"""MapBuilder.reset_envs in a vectorised loop whose episodes end at different steps, at BASELINE config-4 geometry
(480x640 depth -> 400x400 local maps at 3 cm, the bench.BuilderWorkload walk): one JSON line per arm and case.

Environment e runs 100-step episodes offset by e * 100 / b steps, so an environment ends every few steps; its pose and
depth frame at step t are those of step (t + offset) % 100 of its own walk.  Cases: 32 environments with height maps,
and 8 environments with 16 classes given as class ids (label_map=, num_classes=).  Arms, alternated in one process:
  A  reset_envs(done) with the done flags in a CUDA bool tensor (no host sync);
  B  the hand edit it replaces, top[done] = fill; mask[done] = False (heights[done] = -inf for value maps), indexed with
     the same CUDA flags and done only on steps where an episode ends; the in-place edit drops the tracked box and
     rectangles, so the next merge scans the whole world map and copies it cell by cell;
  C  one batch-1 MapBuilder per environment, reset() when its episode ends.
Each arm warms up over one whole episode (the allocator's cached blocks then serve the timed window) and reports ms per
step, env-steps/s and the peak allocated memory of the timed window.  At the end of every timed window the world maps
of A and B are asserted bit-identical.  A separate torch.profiler pass (CUDA activities) over arm A takes the reset
kernels' time per call.

usage: python scripts/time_reset_envs.py [--steps 100] [--repeat 2] [--profile-steps 30] [--cases all]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
import dungeon_maps_b200 as dmap  # noqa: E402
from dungeon_maps_b200 import synth  # noqa: E402

EPISODE = 100


def card():
  name = torch.cuda.get_device_name(0)
  try:
    limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
  except (OSError, subprocess.SubprocessError):
    limit = "unknown"
  return {"gpu": name, "power_limit": limit or "unknown"}


def make_builder(dev):
  proj = dmap.MapProjector(width=640, height=480, hfov=bench.HFOV, cam_pose=[0., 0., 0.], width_offset=0.,
                           height_offset=0., cam_pitch=bench.PITCH, cam_height=bench.CAM_H, map_res=bench.RES,
                           map_width=bench.MW, map_height=bench.MH, trunc_depth_min=0.15, trunc_depth_max=5.05,
                           clip_border=10, fill_value=dmap.NINF, to_global=True, device=dev)
  return dmap.MapBuilder(map_projector=proj)


class Staggered:
  """One 100-step cycle of the staggered loop: per step the depth frames, poses, class ids and done flags."""

  def __init__(self, B, C, dev):
    self.B, self.C = B, C
    w = bench.BuilderWorkload(argparse.Namespace(scene="room"))
    w.B = B
    poses = w.walk(B, EPISODE, 0)
    frames = w.frames_for(poses, dev, 0)
    off = [e * EPISODE // B for e in range(B)]
    k = [[(t + off[e]) % EPISODE for e in range(B)] for t in range(EPISODE)]
    env = torch.arange(B)
    self.depth = [torch.stack([frames[k[t][e]][e] for e in range(B)]) for t in range(EPISODE)]
    del frames
    self.poses = [poses[torch.tensor(k[t]), env] for t in range(EPISODE)]
    self.done_host = [[k[t][e] == 0 for e in range(B)] for t in range(EPISODE)]
    self.done = [torch.tensor(d, device=dev) for d in self.done_host]
    self.labels = None
    if C:
      pool = [synth.block_labels(B, C, 480, 640, seed=t, device=dev).to(torch.uint8) for t in range(16)]
      self.labels = [pool[t % 16] for t in range(EPISODE)]
    self.local_kw = dict(to_global=False, width_offset=bench.MW / 2., height_offset=0., map_width=bench.MW,
                         map_height=bench.MH)

  def kw(self, t, e=None):
    if not self.C:
      return self.local_kw
    ids = self.labels[t % EPISODE]
    return dict(self.local_kw, label_map=ids if e is None else ids[e:e + 1], num_classes=self.C)


def hand_edit(builder, done):
  wm = builder.world_map
  if wm is None or wm.is_empty:
    return
  wm.topdown_map[done] = dmap.NINF
  wm.mask[done] = False
  if not wm.is_height_map:
    wm.height_map[done] = dmap.NINF


class Arm:
  def __init__(self, name, loop, dev):
    self.name, self.loop, self.dev = name, loop, dev
    self.builders = [make_builder(dev) for _ in range(loop.B)] if name == "C" else [make_builder(dev)]

  def step(self, t):
    lp, i = self.loop, t % EPISODE
    if self.name == "C":
      for e, bld in enumerate(self.builders):
        if t > 0 and lp.done_host[i][e]:
          bld.reset()
        bld.step(lp.depth[i][e:e + 1], cam_pose=lp.poses[i][e:e + 1], **lp.kw(i, e))
      return
    bld = self.builders[0]
    if t > 0:
      if self.name == "A":
        bld.reset_envs(lp.done[i])
      elif any(lp.done_host[i]):
        hand_edit(bld, lp.done[i])
    bld.step(lp.depth[i], cam_pose=lp.poses[i], **lp.kw(i))


def time_arm(arm, args):
  for t in range(EPISODE):
    arm.step(t)
  torch.cuda.synchronize()
  dev = arm.dev
  torch.cuda.reset_peak_memory_stats(dev)
  base = torch.cuda.memory_allocated(dev)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  h0 = time.perf_counter()
  e0.record()
  for t in range(EPISODE, EPISODE + args.steps):
    arm.step(t)
  e1.record()
  torch.cuda.synchronize()
  host_s = time.perf_counter() - h0
  ms = e0.elapsed_time(e1) / args.steps
  lp = arm.loop
  return {"arm": arm.name, "envs": lp.B, "classes": lp.C or None, "maps": "class ids" if lp.C else "height",
          "steps": args.steps, "warmup_steps": EPISODE, "ms_per_step": round(ms, 4),
          "env_steps_per_s": round(lp.B / ms * 1e3, 1), "host_wall_ms_per_step": round(host_s * 1e3 / args.steps, 4),
          "peak_allocated_bytes": int(torch.cuda.max_memory_allocated(dev) - base),
          "world_shape_at_end": list(arm.builders[0].world_map.mask.shape)}


def assert_same_world(a, b):
  wa, wb = a.builders[0].world_map, b.builders[0].world_map
  assert wa.mask.shape == wb.mask.shape, (wa.mask.shape, wb.mask.shape)
  for name in ("width_offset", "height_offset"):
    assert float(getattr(wa.proj, name)) == float(getattr(wb.proj, name)), name
  for x, y in ((wa.topdown_map, wb.topdown_map), (wa.height_map, wb.height_map)):
    assert torch.equal(x.contiguous().view(torch.int32), y.contiguous().view(torch.int32)), "world maps differ"
  assert torch.equal(wa.mask, wb.mask), "world masks differ"


def profile_resets(loop, dev, args):
  from torch.profiler import ProfilerActivity, profile
  arm = Arm("A", loop, dev)
  for t in range(EPISODE):
    arm.step(t)
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for t in range(EPISODE, EPISODE + args.profile_steps):
      arm.step(t)
    torch.cuda.synchronize()
  us, calls = defaultdict(float), defaultdict(int)
  for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
      us[e.name] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
      calls[e.name] += 1
  short = lambda k: k.split("(")[0].replace("void ", "").replace("dm::", "")
  resets = {short(k): {"us_per_call": round(v / calls[k], 2), "calls": calls[k]}
            for k, v in us.items() if "fuse_clear" in k}
  return {"profile": "arm A reset kernels", "envs": loop.B, "classes": loop.C or None, "steps": args.profile_steps,
          "reset_kernels": resets,
          "all_kernels_us_per_step": round(sum(us.values()) / args.profile_steps, 1)}


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--steps", type=int, default=100, help="timed steps per arm, after one whole episode of warm-up")
  ap.add_argument("--repeat", type=int, default=2)
  ap.add_argument("--profile-steps", type=int, default=30)
  ap.add_argument("--cases", default="all", help="all | height | labels")
  args = ap.parse_args()
  if args.steps < 1 or args.repeat < 1 or args.profile_steps < 1:
    ap.error("--steps, --repeat and --profile-steps must be >= 1")
  if not torch.cuda.is_available():
    sys.exit("time_reset_envs.py measures on a CUDA device; none is available")
  dev = torch.device("cuda", 0)
  print(json.dumps(card()), flush=True)
  cases = [(32, 0), (8, 16)]
  if args.cases == "height":
    cases = cases[:1]
  elif args.cases == "labels":
    cases = cases[1:]
  for B, C in cases:
    loop = Staggered(B, C, dev)
    for _ in range(args.repeat):
      arms = {}
      for name in ("A", "B", "C"):
        arms[name] = Arm(name, loop, dev)
        print(json.dumps(time_arm(arms[name], args)), flush=True)
        if name == "C":
          del arms["C"]
      assert_same_world(arms["A"], arms["B"])
      print(json.dumps({"check": "A and B world maps bit-identical", "envs": B, "classes": C or None}), flush=True)
      del arms
    print(json.dumps(profile_resets(loop, dev, args)), flush=True)
    del loop
    torch.cuda.empty_cache()


if __name__ == "__main__":
  main()
