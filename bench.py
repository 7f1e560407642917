#!/usr/bin/env python
"""bench.py — top-down maps/sec of the fused projection (BASELINE.json config 2), plus the other
workloads of the path as separately labelled lines.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload proj|flow|builder|builder_fixed|proj5] [--scene room|iid] [--dump-outputs DIR]

Default (`--workload proj`, the line the driver reads): one "step" = one pass of the hot path
(dm_orth_project_f32: fused projection + resolve) over one batch of 64 synthetic 480x640 depth frames
+ 16 one-hot float32 semantic channels → 400x400 local maps (topdown, mask, height); every step takes the next of 4
different input batches and a fresh pose set.  `e2e` of that line is the same workload from HOST buffers with the
semantics given as uint8 class ids (dm_orth_project_labels_host_f32: bit-identical outputs, 5 instead of 68 bytes per
pixel across PCIe); `e2e_float32` is the float32-plane host entry.  The same JSON line carries, under `extra`, the
other named configurations (timed outside the headline region) and, under `pcie`, every rank's pinned-copy rates.
Other workloads (BASELINE.json configs 3, 4, 5; `--workload X` makes one of them the line):
  proj_labels    config 2 with the semantics as class ids (label_map=, num_classes=16), device-resident
  flow           camera_affine_grid, 256 x 480x640 frames, fresh random pose deltas every step
  builder        MapBuilder.step (plot + reference-parity merge), 32 environments walking for 100 steps
  builder_fixed  the same walk merged in place into fixed 2400x2400 world canvases (opt-in mode)
  proj5          the projection at 1280x720 with 40 semantic channels, 8 different 64-frame chunks in rotation
  proj5_labels   the same with class ids
  proj5_job      config 5 as a job: 4096 / N frames per rank streamed from host memory in 64-frame chunks (class ids)
N > 1: one process per GPU (torchrun; `python bench.py --gpus N` on its own re-launches itself that way), every
rank works on its own environments, no collective on the data path (weak scaling).  Prints ONE JSON line on rank 0.
--dump-outputs DIR: after the timed steps, rank 0 writes the arrays its last timed step returned as DIR/<name>.npy
(see dump_outputs); the inputs depend on the arguments only, so two builds can be compared file by file.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree, which may be read-only

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import numpy as np
import torch

HFOV, PITCH, CAM_H, RES = math.radians(70), math.radians(-10), 0.88, 0.03
MH, MW = 400, 400


class ClockSampler:
  """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
  FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
            "clocks_event_reasons.sw_power_cap")

  def __init__(self, gpu_index: int):
    self.rows, self.proc = [], None
    try:
      self.proc = subprocess.Popen(
        ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(gpu_index)],
        stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.t = threading.Thread(target=self._pump, daemon=True)
      self.t.start()
    except Exception:
      self.proc = None

  def _pump(self):
    for line in self.proc.stdout:
      self.rows.append((time.perf_counter(), line.strip()))

  def wait_ready(self, timeout: float = 3.0) -> None:
    """nvidia-smi needs a moment before its first sample; short timed regions would otherwise see none."""
    t_end = time.perf_counter() + timeout
    while self.proc is not None and not self.rows and time.perf_counter() < t_end:
      time.sleep(0.01)

  def stop(self, t0: float, t1: float) -> dict:
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    inside = [r for (t, r) in self.rows if t0 <= t <= t1] or [r for (_, r) in self.rows[-3:]]
    sm, smax, reasons = [], [], set()
    names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
    for r in inside:
      f = [x.strip() for x in r.split(",")]
      try:
        sm.append(float(f[0])); smax.append(float(f[1]))
      except Exception:
        continue
      for n, v in zip(names, f[3:7]):
        if v.lower().startswith("active"):
          reasons.add(n)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  try:
    with open(path) as f:
      return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
  except Exception:
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(key: str):
  """dram bytes per launch of the workload's dominant kernel from the committed ncu --set full summary."""
  try:
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
      d = json.load(f)
    if key == "proj":
      return d.get("dram_bytes_per_step")
    return (d.get(key) or {}).get("dram_bytes_per_step")
  except Exception:
    return None


def intrinsics(W, H):
  cx, cy = W / 2., H / 2.
  fx = cx / np.tan(HFOV / 2.)
  return fx, fx, cx, cy


# ================================================================================================
# Workloads.  Each one: setup(dev, rank) once; step() = one pass over one batch on the device;
# e2e_setup()/e2e_step() = the same pass from pinned HOST buffers with the copies inside;
# cpu_step(threads) -> units processed by one bounded CPU pass of the oracle port.
# ================================================================================================

class ProjWorkload:
  """BASELINE config 2 (and config 5's shapes with key='proj5')."""
  unit = "maps/s"
  kernel = "dm::proj_ws_kernel (one step = ONE persistent launch of dm_orth_project_f32: projection + resolve)"

  def __init__(self, args, key="proj"):
    self.key, self.scene = key, args.scene
    self.labels = key.endswith("_labels")
    key = key.replace("_labels", "")
    if key == "proj":
      self.B, self.H, self.W, self.C = 64, 480, 640, 16
      self.metric = "top-down maps/sec (batch 64, 640x480 depth + 16 semantic channels -> 400x400 maps)"
      self.name = ("BASELINE config 2: 64 x 480x640 depth + 16-channel one-hot semantics -> 400x400 maps "
                   "(topdown + mask + height), per GPU")
    else:
      self.B, self.H, self.W, self.C = 64, 720, 1280, 40
      self.metric = "top-down maps/sec (1280x720 depth + 40 semantic channels -> 400x400 maps, 64-frame chunks)"
      self.name = ("BASELINE config 5 (steady state of the 4096-frame job): one 64-frame chunk of 1280x720 depth + "
                   "40-channel one-hot semantics -> 400x400 maps per step, per GPU; every GPU streams 4096/N frames")
    self.sets = 8 if key == "proj5" else 4
    self.units_per_step = self.B
    # SURVEY.md §8d: read 4*N*(1+C) input bytes, write Mh*Mw*(4C + C + 4) output bytes per frame
    in_bytes = self.H * self.W * (5 if self.labels else 4 * (1 + self.C))
    self.algo_bytes_per_step = self.B * (in_bytes + MH * MW * (4 * self.C + self.C + 4))
    self.l2_note = (f"{self.algo_bytes_per_step / 1e9:.2f} GB move per step (inputs {self.B * in_bytes / 1e9:.2f} GB), larger than "
                    "the 126 MB L2; no flush needed")
    if self.labels:
      self.kernel = "dm::proj_lbl_kernel (one step = ONE persistent launch of dm_orth_project_labels_f32)"
      self.metric += " [semantics given as uint8 class ids]"
      self.name += "; semantics enter as (b,1,H,W) uint8 class ids (label_map=, num_classes=16): bit-identical outputs"

  def kwargs(self):
    fx, fy, cx, cy = intrinsics(self.W, self.H)
    return dict(map_res=RES, map_width=MW, map_height=MH, focal_x=fx, focal_y=fy, center_x=cx, center_y=cy,
                trunc_depth_min=0.15, trunc_depth_max=5.05, trunc_height_max=None, clip_border=10,
                to_global=False, flip_h=True, fill_value=-np.inf, reduction=None, get_height_map=True)

  def config(self, world):
    return {"workload": self.name, "scene": self.scene, "fill_value": "-inf", "frames_per_step_per_gpu": self.B,
            "input_rotation": f"{self.sets} different input batches in rotation, a fresh pose set every step",
            "parallelism": f"batch-sharded x{world}, no collective", "l2": self.l2_note}

  def setup(self, dev, rank):
    import dungeon_maps_b200 as dmap
    from dungeon_maps_b200 import synth
    self.dev = dev
    # a real caller never projects the same tensors twice: `sets` different input batches in rotation, and a pose
    # set of its own for every step (the parameter caches of the host layer see fresh poses)
    self.batches = []
    for i in range(self.sets):
      seed = rank * 64 + i
      depth, _, _ = synth.frames(self.scene, self.B, self.H, self.W, 0, seed=seed, device=dev)
      ids = synth.block_labels(self.B, self.C, self.H, self.W, seed, device=dev)   # the ids block_onehot expands
      values = None if self.labels else synth.block_onehot(self.B, self.C, self.H, self.W, seed, device=dev)
      self.batches.append((depth, values, ids.to(torch.uint8)))
    self.depth, self.values, self.label_ids = self.batches[0]
    self.pose_sets = [synth.poses(self.B, 7919 * rank + i) for i in range(257)]
    self.t = 0
    self.proj = dmap.MapProjector(width=self.W, height=self.H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=200.,
                                  height_offset=0., cam_pitch=PITCH, cam_height=CAM_H, map_res=RES, map_width=MW,
                                  map_height=MH, trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=10,
                                  to_global=False, fill_value=dmap.NINF, device=dev)
    self.pose_host = self.pose_sets[0]

  def step(self):
    depth, values, ids = self.batches[self.t % self.sets]
    pose = self.pose_sets[self.t % len(self.pose_sets)]
    self.t += 1
    if self.labels:
      self.out = self.proj.orth_project(depth, cam_pose=pose, get_height_map=True, label_map=ids,
                                        num_classes=self.C)
    else:
      self.out = self.proj.orth_project(depth, values, cam_pose=pose, get_height_map=True)
    self.last = (depth, values, ids, pose)
    return self.out

  def outputs(self):
    top, mask, hgt = self.out
    return {"topdown": top, "mask": mask, "height": hgt}

  def e2e_setup(self, float32=False):
    """Host-buffer leg.  Default: semantics as uint8 class ids (what a segmentation network emits and what the
    reference's object-map demo starts from, demos/object_map/run.py:117-124); float32=True: the one-hot float32
    planes the reference's orth_project signature takes."""
    B, C = self.B, self.C
    depth, values, ids = self.batches[0]
    self.h_depth = depth.cpu().pin_memory().numpy()
    self.e2e_float = bool(float32) and not self.labels
    if self.e2e_float:
      self.h_values = values.cpu().pin_memory().numpy()
    else:
      self.h_values = ids.cpu().pin_memory().numpy()
    if not hasattr(self, "o_top"):
      self.o_top = torch.empty((B, C, MH, MW), dtype=torch.float32).pin_memory().numpy()
      self.o_mask = torch.empty((B, C, MH, MW), dtype=torch.uint8).pin_memory().numpy()
      self.o_hgt = torch.empty((B, 1, MH, MW), dtype=torch.float32).pin_memory().numpy()
    self.h2d = self.h_depth.nbytes + self.h_values.nbytes + B * 192
    self.d2h = self.o_top.nbytes + self.o_mask.nbytes + self.o_hgt.nbytes
    self.e2e_path = ("hostapi.orth_project_host -> dm_orth_project_host_f32 (pinned host buffers, float32 one-hot planes)"
                     if self.e2e_float else
                     "hostapi.orth_project_host(label_map=uint8 class ids, num_classes=%d) -> "
                     "dm_orth_project_labels_host_f32 (pinned host buffers; outputs bit-identical to the float32-plane entry)" % C)

  def e2e_step(self):
    from dungeon_maps_b200 import hostapi
    if self.e2e_float:
      hostapi.orth_project_host(self.h_depth, self.h_values, None, self.pose_host, 200., 0., PITCH, CAM_H,
                                device=self.dev.index, out=(self.o_top, self.o_mask, self.o_hgt), **self.kwargs())
    else:
      hostapi.orth_project_host(self.h_depth, None, None, self.pose_host, 200., 0., PITCH, CAM_H,
                                device=self.dev.index, out=(self.o_top, self.o_mask, self.o_hgt),
                                label_map=self.h_values, num_classes=self.C, **self.kwargs())

  def e2e_check(self):
    depth, values, ids = self.batches[0]
    if self.labels:
      want = self.proj.orth_project(depth, cam_pose=self.pose_host, get_height_map=True, label_map=ids,
                                    num_classes=self.C)
    else:  # the device-resident float32 path is the yardstick for both host entries
      want = self.proj.orth_project(depth, values, cam_pose=self.pose_host, get_height_map=True)
    assert np.array_equal(self.o_top, want[0].cpu().numpy()) and \
        np.array_equal(self.o_mask, want[1].cpu().numpy().view(np.uint8)) and \
        np.array_equal(self.o_hgt, want[2][:, :1].cpu().numpy()), "host-buffer path and device path disagree"

  def cpu_setup(self, threads):
    from dungeon_maps_b200 import synth
    from oracle import dm_oracle as orc
    n = min(self.B, max(threads, 8))  # bounded sample: one frame per host thread, at most the batch
    depth, values, pose = synth.frames(self.scene, n, self.H, self.W, self.C, seed=0)
    d, v, p = depth.numpy(), values.numpy(), pose.numpy()
    kw = self.kwargs()
    orc.orth_project(d[:1], v[:1], None, p[:1], 200., 0., PITCH, CAM_H, threads=1, **kw)  # page-in
    self.cpu_units = n
    self.cpu_fn = lambda: orc.orth_project(d, v, None, p, 200., 0., PITCH, CAM_H, threads=threads, **kw)
    self.cpu_sample = (f"{n} frames per pass of the same workload ({self.scene} scene), oracle/dm_oracle.c "
                       f"(scalar C restatement of the reference CPU path) with {threads} OpenMP threads")


  def ref_setup(self, threads):
    """The UNMODIFIED reference (dungeon_maps v0.0.3a1, pure Python + torch) through oracle/ref_shim.py — the
    12-line torch_scatter stand-in — applied per sample (it raises for batch > 1, utils.py:311-316)."""
    from dungeon_maps_b200 import synth
    from oracle import ref_shim
    ref = ref_shim.load_reference()
    torch.set_num_threads(threads)
    n = 8  # bounded sample: 8 frames per pass (≈ 50 ms each on a 16-thread host)
    depth, values, pose = synth.frames(self.scene, n, self.H, self.W, self.C, seed=0)
    proj = ref.MapProjector(width=self.W, height=self.H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=200.,
                            height_offset=0., cam_pitch=PITCH, cam_height=CAM_H, map_res=RES, map_width=MW,
                            map_height=MH, trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=10,
                            to_global=False, fill_value=-np.inf)

    def one_pass():
      for i in range(n):
        proj.orth_project(depth_map=depth[i:i + 1], value_map=values[i:i + 1], cam_pose=pose[i:i + 1],
                          get_height_map=True)
    self.cpu_units = n
    self.cpu_fn = one_pass
    self.cpu_sample = (f"{n} frames per pass of the same workload ({self.scene} scene), the unmodified reference "
                       f"(MapProjector.orth_project per sample, torch {torch.__version__} CPU, {threads} threads, "
                       "torch_scatter replaced by the scatter_reduce_ stand-in of oracle/ref_shim.py)")


class FlowWorkload:
  """BASELINE config 3: compute_ego_flow / camera_affine_grid, batch 256 x 480x640, random pose deltas."""
  unit = "frames/s"
  key = "flow"
  kernel = "dm::flow_kernel (one step = one launch of dm_affine_grid_f32)"
  metric = "ego-flow frames/sec (camera_affine_grid, batch 256, 640x480 depth, random camera pose deltas)"

  def __init__(self, args):
    self.B, self.H, self.W = 256, 480, 640
    self.scene = args.scene
    self.units_per_step = self.B
    self.algo_bytes_per_step = self.B * self.H * self.W * 12  # SURVEY.md §8d: 4 B in, 8 B out per pixel
    self.name = "BASELINE config 3: camera_affine_grid on 256 x 480x640 depth frames, random pose deltas, per GPU"

  def config(self, world):
    return {"workload": self.name, "scene": self.scene, "frames_per_step_per_gpu": self.B,
            "input_rotation": "a fresh set of 256 pose deltas every step",
            "parallelism": f"batch-sharded x{world}, no collective",
            "l2": "0.94 GB moved per step, larger than the 126 MB L2; no flush needed"}

  def _deltas(self, n, seed, device=None):
    from dungeon_maps_b200 import synth
    u = synth.uniform((n, 3), seed ^ 0xF10, -1.0, 1.0, device)
    return u * torch.tensor([0.25, 0.25, 0.3], dtype=torch.float32, device=device)  # SURVEY.md §8d

  def setup(self, dev, rank):
    import dungeon_maps_b200 as dmap
    from dungeon_maps_b200 import synth
    self.dev = dev
    self.depth, _, _ = synth.frames(self.scene, self.B, self.H, self.W, 0, seed=rank, device=dev)
    self.delta_sets = [self._deltas(self.B, 104729 * rank + i).cpu() for i in range(257)]  # a fresh set every step
    self.delta_host = self.delta_sets[0]
    self.t = 0
    self.proj = dmap.MapProjector(width=self.W, height=self.H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=0.,
                                  height_offset=0., cam_pitch=PITCH, cam_height=CAM_H, map_res=RES, map_width=MW,
                                  map_height=MH, device=dev)

  def step(self):
    self.out = self.proj.camera_affine_grid(self.depth, self.delta_sets[self.t % len(self.delta_sets)])
    self.t += 1
    return self.out

  def outputs(self):
    return {"grid": self.out}

  def e2e_setup(self):
    self.h_depth = self.depth.cpu().pin_memory()
    self.o_grid = torch.empty((self.B, 1, self.H, self.W, 2), dtype=torch.float32).pin_memory()
    self.h2d = self.h_depth.numel() * 4 + self.B * 192
    self.d2h = self.o_grid.numel() * 4
    self.e2e_path = ("hostapi.camera_affine_grid_host -> MapProjector.camera_affine_grid on pinned host tensors "
                     "(32-frame chunks: H2D copy, kernel, D2H copy of the grid on three streams)")

  def e2e_step(self):
    from dungeon_maps_b200 import hostapi
    hostapi.camera_affine_grid_host(self.proj, self.h_depth, self.delta_host, out=self.o_grid)

  def e2e_check(self):
    want = self.proj.camera_affine_grid(self.depth, self.delta_host)
    assert torch.equal(self.o_grid.nan_to_num(), want.cpu().nan_to_num()), "host path and device path disagree"

  def cpu_setup(self, threads):
    from dungeon_maps_b200 import synth
    from oracle import dm_oracle as orc
    n = min(self.B, max(4 * threads, 16))
    depth, _, _ = synth.frames(self.scene, n, self.H, self.W, 0, seed=0)
    d, p = depth.numpy(), self._deltas(n, 0).numpy()
    fx, fy, cx, cy = intrinsics(self.W, self.H)
    self.cpu_units = n
    self.cpu_fn = lambda: orc.camera_affine_grid(d, p, PITCH, CAM_H, fx, fy, cx, cy, threads=threads)
    self.cpu_sample = f"{n} frames per pass ({self.scene} scene), oracle/dm_oracle.c with {threads} OpenMP threads"


class BuilderWorkload:
  """BASELINE config 4: MapBuilder global fusion, 32 environments, 400x400 local height maps merged into
  the world maps over a 100-step walk.  key='builder': the reference's merge (fuse_topdown_maps: re-scatter
  into a freshly sized canvas every step, one host sync).  key='builder_fixed': opt-in in-place merge
  into fixed 2400x2400 canvases (no reference equivalent, SURVEY.md D5)."""
  unit = "env-steps/s"
  EPISODE = 100
  e2e_min_steps = 50

  def __init__(self, args, key="builder"):
    self.key = key
    self.B, self.H, self.W = 32, 480, 640
    self.units_per_step = self.B
    self.fixed = key == "builder_fixed"
    self.metric = ("MapBuilder env-steps/sec (32 envs, 480x640 depth -> 400x400 local height map -> merged into "
                   + ("fixed 2400x2400 world maps in place)" if self.fixed else "the growing world map, reference semantics)"))
    self.kernel = ("one MapBuilder.step = dm_builder_step_fixed: dm::hmap_proj_kernel + dm::hmap_resolve_kernel + dm::fuse_scatter_kernel (in place)"
                   if self.fixed else
                   "one MapBuilder.step = dm_builder_plot + dm_builder_merge: dm::hmap_proj_kernel, hmap_resolve, fuse_bbox, [host sync], "
                   "fuse_fill, fuse_scatter x2; roofline over the WHOLE step (host sync included)")
    self.name = ("BASELINE config 4: MapBuilder.step over 32 envs x 100-step walk, " +
                 ("fixed 2400x2400 canvases, in-place max-merge" if self.fixed else
                  "fuse_topdown_maps semantics (data-dependent canvas, batch-wide bounding box)"))
    self.t = 0
    self.algo_bytes_total = 0

  def config(self, world):
    return {"workload": self.name, "scene": "room (66 m hall, 32 walkers)", "envs_per_gpu": self.B,
            "episode_steps": self.EPISODE, "world_cells_at_end": getattr(self, "world_shape", None),
            "input_rotation": "every step has its own depth frames and poses (100-step walk)",
            "warmup": "one whole episode (the allocator's cached blocks serve the timed one, like any episode after the first)",
            "parallelism": f"environment-sharded x{world}, no collective",
            "l2": "world maps (>1 GB per step) are larger than the 126 MB L2; no flush needed"}

  @staticmethod
  def walk(b, steps, seed, half=30.0):
    """(steps, b, 3) poses: discrete walk like the reference sim (sim/dungeon.py:244-255): forward 0.25 m / turn ±30°."""
    from dungeon_maps_b200 import synth
    pose = synth.poses(b, seed, xz=half).numpy().astype(np.float64)
    act = (synth.hash_u24(steps * b, seed ^ 0xAC7).numpy() % 4).reshape(steps, b)
    out = np.zeros((steps, b, 3), np.float32)
    for t in range(steps):
      out[t] = pose
      fwd = act[t] < 2
      pose[:, 0] += np.where(fwd, 0.25 * np.sin(pose[:, 2]), 0.0)
      pose[:, 1] += np.where(fwd, 0.25 * np.cos(pose[:, 2]), 0.0)
      pose[:, 2] += np.where(act[t] == 2, math.radians(30), 0.0) - np.where(act[t] == 3, math.radians(30), 0.0)
      pose[:, :2] = np.clip(pose[:, :2], -half, half)
    return torch.from_numpy(out)

  def frames_for(self, poses, dev, seed):
    from dungeon_maps_b200 import synth
    return [synth.room_depth(poses.shape[1], self.H, self.W, HFOV, PITCH, CAM_H, poses[t] if dev is None else poses[t].to(dev), seed, half=33.0,
                             device=dev) for t in range(poses.shape[0])]

  def make_builder(self, dev):
    import dungeon_maps_b200 as dmap
    proj = dmap.MapProjector(width=self.W, height=self.H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=0.,
                             height_offset=0., cam_pitch=PITCH, cam_height=CAM_H, map_res=RES, map_width=MW,
                             map_height=MH, trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=10,
                             fill_value=dmap.NINF, to_global=True, device=dev)
    if self.fixed:
      return dmap.MapBuilder(map_projector=proj, fixed_canvas=(2400, 2400))
    return dmap.MapBuilder(map_projector=proj)

  def setup(self, dev, rank, frames=None):
    self.dev = dev
    self.poses = self.walk(self.B, self.EPISODE, rank)
    self.frames = frames if frames is not None else self.frames_for(self.poses, dev, rank)
    self.builder = self.make_builder(dev)
    self.local_kw = dict(to_global=False, width_offset=MW / 2., height_offset=0., map_width=MW, map_height=MH)

  def step(self):
    t = self.t % self.EPISODE
    if t == 0:
      # a new episode: the loop lets go of the last episode's world map before it builds the next one (held across the
      # reset it keeps 0.9 GB of fixed canvases alive and the new episode's canvases cost a 75 ms cudaMalloc, once)
      self.out = None
      self.builder.reset()
    before = self.builder.world_map
    cells = lambda m: 0 if m is None or m.is_empty else m.mask.numel()
    n_before = cells(before)
    local = self.builder.step(self.frames[t], cam_pose=self.poses[t], **self.local_kw)
    after = self.builder.world_map
    # plot: read the depth frames, write (height f32 + mask u8) of the local maps (SURVEY.md §8d, C = 0)
    self.algo_bytes_total += self.B * (4 * self.H * self.W + 5 * MH * MW)
    if self.fixed:  # merge in place: read the local maps, read-modify-write the cells they touch
      self.algo_bytes_total += 5 * local.mask.numel() + 8 * int(local.mask.shape[0]) * MH * MW
    else:           # read (height f32 + mask u8) of both sources, write (height f32 + mask u8) of the new world
      self.algo_bytes_total += 5 * (n_before + cells(local)) + 5 * cells(after)
    self.world_shape = list(after.mask.shape)
    self.t += 1
    self.out, self.local = after, local
    return after

  def outputs(self):
    """The local map MapBuilder.step returned and the world map it merged that map into (height maps: C = 0)."""
    w, l = self.out, self.local
    return {"world_height": w.topdown_map, "world_mask": w.mask, "world_width_offset": w.proj.width_offset,
            "world_height_offset": w.proj.height_offset, "local_height": l.topdown_map, "local_mask": l.mask}

  def reset_counters(self):
    self.algo_bytes_total = 0

  def e2e_setup(self):
    self.h_frames = [f.cpu().pin_memory() for f in self.frames[:10]]
    self.e2e_builder = self.make_builder(self.dev)
    self.h2d = self.h_frames[0].numel() * 4 + self.B * 464
    self.d2h = 40  # the merge's bounding box; the world map stays on the device, like the reference's
    self.e2e_t = 0
    self.e2e_path = "MapBuilder.step on pinned host depth (H2D copy, plot, merge incl. its bbox D2H sync)"

  def e2e_step(self):
    t = self.e2e_t % len(self.h_frames)
    if t == 0:
      self.e2e_builder.reset()
    d = self.h_frames[t].to(self.dev, non_blocking=True)
    self.e2e_builder.step(d, cam_pose=self.poses[t], **self.local_kw)
    torch.cuda.current_stream(self.dev).synchronize()
    self.e2e_t += 1

  def e2e_check(self):
    """Two environments of this walk, 12 steps, through a MapBuilder of their own on the GPU and through the
    oracle (plot via oracle/dm_oracle.c, merge via the restatement of fuse_topdown_maps): identical final world
    maps (shape, offsets, sha256 of heights and mask)."""
    import hashlib
    from oracle import dm_oracle as orc
    n, T = 2, 12
    fx, fy, cx, cy = intrinsics(self.W, self.H)
    builder = self.make_builder(self.dev)
    world = None
    for t in range(T):
      depth = self.frames[t][:n].contiguous()
      p = self.poses[t][:n]
      builder.step(depth, cam_pose=p, **self.local_kw)
      if self.fixed:
        continue
      top, mask, hgt = orc.orth_project(depth.cpu().numpy(), None, None, p.numpy(), MW / 2., 0., PITCH, CAM_H, RES, MW,
                                        MH, fx, fy, cx, cy, 0.15, 5.05, None, 10, False, True, -np.inf, None, True,
                                        threads=os.cpu_count() or 1)
      src = [orc.FuseSource(hgt, mask, None, MW / 2., 0., RES, True, False, p.numpy())]
      if world is not None:
        src.insert(0, orc.FuseSource(world["height"], world["mask"], None, world["width_offset"],
                                     world["height_offset"], RES, True, True, p.numpy()))
      world = orc.fuse(src, True, p.numpy(), RES, True) or world
    wm = builder.world_map
    if self.fixed:  # no reference semantics to compare with: the canvas must hold what a second builder produces
      again = self.make_builder(self.dev)
      for t in range(T):
        again.step(self.frames[t][:n].contiguous(), cam_pose=self.poses[t][:n], **self.local_kw)
      assert torch.equal(wm.topdown_map, again.world_map.topdown_map) and torch.equal(wm.mask, again.world_map.mask)
      return
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    assert [wm.proj.map_height, wm.proj.map_width] == [world["map_height"], world["map_width"]], "world shape"
    assert float(wm.proj.width_offset) == float(np.float32(world["width_offset"])), "world width offset"
    assert sha(wm.topdown_map.cpu().numpy()) == sha(world["topdown"]), "world heights differ from the oracle"
    assert sha(wm.mask.cpu().numpy()) == sha(world["mask"].astype(bool)), "world mask differs from the oracle"

  def cpu_setup(self, threads):
    from oracle import dm_oracle as orc
    n, T = 2, 4
    poses = self.walk(n, T, 0)
    frames = [f.numpy() for f in self.frames_for(poses, None, 0)]
    fx, fy, cx, cy = intrinsics(self.W, self.H)

    def episode():
      world = None
      for t in range(T):
        p = poses[t].numpy()
        top, mask, hgt = orc.orth_project(frames[t], None, None, p, MW / 2., 0., PITCH, CAM_H, RES, MW, MH, fx, fy, cx,
                                          cy, 0.15, 5.05, None, 10, False, True, -np.inf, None, True, threads=threads)
        src = [orc.FuseSource(hgt, mask, None, MW / 2., 0., RES, True, False, p)]
        if world is not None:
          src.insert(0, orc.FuseSource(world["height"], world["mask"], None, world["width_offset"],
                                       world["height_offset"], RES, True, True, p))
        world = orc.fuse(src, True, p, RES, True) or world
    self.cpu_units = n * T
    self.cpu_fn = episode
    self.cpu_sample = (f"{n} envs x {T} steps per pass (plot via oracle/dm_oracle.c with {threads} threads, merge via the "
                       f"numpy restatement of fuse_topdown_maps)")


def proj5_job(dev, rank, world, barrier, max_over_ranks):
  """BASELINE config 5 as the job it names: 4096 frames of 1280x720 depth + 40-class semantics, 4096 / N per rank,
  HOST-resident inputs (uint8 class ids: the float32 planes of 4096 frames would be 619 GB), streamed through
  dm_orth_project_labels_host_f32 in 64-frame chunks — 8 different chunks in rotation — with the results landing in
  pinned host memory.  Steady state of the whole job, PCIe inside."""
  from dungeon_maps_b200 import hostapi, synth
  B, H, W, C, distinct = 64, 720, 1280, 40, 8
  frames = 4096 // world
  chunks = max(frames // B, 1)
  h_depth, h_ids, poses = [], [], []
  for i in range(min(distinct, chunks)):
    seed = 4096 + rank * 64 + i
    d, _, pose = synth.frames("room", B, H, W, 0, seed=seed, device=dev)
    h_depth.append(d.cpu().pin_memory().numpy())
    h_ids.append(synth.block_labels(B, C, H, W, seed, device=dev).to(torch.uint8).cpu().pin_memory().numpy())
    poses.append(pose.cpu())
    del d
  out = (torch.empty((B, C, MH, MW), dtype=torch.float32).pin_memory().numpy(),
         torch.empty((B, C, MH, MW), dtype=torch.uint8).pin_memory().numpy(),
         torch.empty((B, 1, MH, MW), dtype=torch.float32).pin_memory().numpy())
  fx, fy, cx, cy = intrinsics(W, H)
  kw = dict(map_res=RES, map_width=MW, map_height=MH, focal_x=fx, focal_y=fy, center_x=cx, center_y=cy,
            trunc_depth_min=0.15, trunc_depth_max=5.05, trunc_height_max=None, clip_border=10, to_global=False,
            flip_h=True, fill_value=-np.inf, reduction=None, get_height_map=True)

  def chunk(i):
    k = i % len(h_depth)
    hostapi.orth_project_host(h_depth[k], None, None, poses[k], 200., 0., PITCH, CAM_H, device=dev.index, out=out,
                              label_map=h_ids[k], num_classes=C, **kw)
  chunk(0)
  barrier()
  t0 = time.perf_counter()
  for i in range(chunks):
    chunk(i)
  torch.cuda.synchronize(dev)
  el = max_over_ranks(time.perf_counter() - t0)
  h2d = (h_depth[0].nbytes + h_ids[0].nbytes) * chunks
  d2h = sum(o.nbytes for o in out) * chunks
  return {"value": world * chunks * B / el, "unit": "maps/s", "frames_per_rank": chunks * B, "chunks_per_rank": chunks,
          "distinct_chunks": len(h_depth), "seconds": el, "h2d_gbs_per_rank": h2d / el / 1e9,
          "d2h_gbs_per_rank": d2h / el / 1e9,
          "workload": "BASELINE config 5 as a job: 4096 x (1280x720 depth + 40-class uint8 ids) -> 400x400 maps "
                      "(topdown f32 x40, mask x40, height), host-resident inputs and outputs, 64-frame chunks"}


def make_workload(args, key=None):
  key = key or args.workload
  if key in ("proj", "proj5", "proj_labels", "proj5_labels"):
    return ProjWorkload(args, key)
  if key == "flow":
    return FlowWorkload(args)
  return BuilderWorkload(args, key)


# ================================================================================================

DUMP_BYTES = 48 << 20  # all files of one --dump-outputs directory together


def dump_positions(numel: int, k: int) -> np.ndarray:
  """Sorted distinct flat positions, at most k of numel, of a dumped sample: seeded, so the same for the same shape."""
  return np.unique(np.random.default_rng(0).integers(0, numel, size=k))


def dump_outputs(arrays: dict, out_dir: str) -> None:
  """Writes every array as out_dir/<name>.npy, float64 as float64 and anything else as float32 (masks as 0 / 1), with
  finite numbers only: a floating-point array also gets out_dir/<name>_nonfinite.npy (0 finite, 1 +inf, -1 -inf,
  2 NaN) and holds 0 where that is not 0, so the -inf fill of unobserved map cells and NaNs survive the dump.  An
  array larger than its share of DUMP_BYTES is written as the 1-D sample of its flattened (row-major) elements at
  dump_positions(numel, k)."""
  os.makedirs(out_dir, exist_ok=True)
  tensors = {name: torch.as_tensor(x).detach() for name, x in arrays.items()}
  share = DUMP_BYTES // sum(2 if t.is_floating_point() else 1 for t in tensors.values())
  for name, t in tensors.items():
    floating = t.is_floating_point()
    dtype = torch.float64 if t.dtype == torch.float64 else torch.float32
    k = share // dtype.itemsize
    if t.numel() > k:
      t = t.reshape(-1)[torch.from_numpy(dump_positions(t.numel(), k)).to(t.device)]
    t = t.to(dtype)
    if floating:
      flag = torch.zeros_like(t).masked_fill_(t == math.inf, 1).masked_fill_(t == -math.inf, -1)
      flag.masked_fill_(t.isnan(), 2)
      np.save(os.path.join(out_dir, name + "_nonfinite.npy"), flag.float().cpu().numpy())
      t = t.masked_fill(flag != 0, 0)
    np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


_RESULT_LINE = []


def _emit(line: str) -> None:
  """The JSON line of this process (printed by main() once fd 1 is the real stdout again)."""
  _RESULT_LINE[:] = [line]


def timed_cpu(wl, threads: int, kind: str, budget_s: float = 20.0):
  """One CPU implementation of the workload (wl.cpu_fn, set up by the caller) on a bounded sample."""
  done, t0 = 0, time.perf_counter()
  while True:
    wl.cpu_fn()
    done += wl.cpu_units
    el = time.perf_counter() - t0
    if el > budget_s / 2 or (el >= 5.0 and done >= 8 * max(wl.units_per_step, wl.cpu_units)):
      break
  return {"value": done / el, "unit": wl.unit, "cores": threads, "kind": kind,
          "sample": f"{wl.cpu_sample}; {done} units in {el:.1f} s"}


def cpu_baseline(wl, threads: int):
  """The oracle port on the same workload: bounded sample (≈10-20 s of CPU work)."""
  wl.cpu_setup(threads)
  return timed_cpu(wl, threads, "port")


def reference_importable() -> bool:
  try:
    from oracle import ref_shim
    return ref_shim.reference_root() is not None
  except Exception:
    return False


def run_reference(args):
  """The reference arm: the reference's own CPU implementation of the path on this box's host cores.  When the
  unmodified reference is importable (baseline/_ref travels to the GPU box) the line's value is ITS throughput
  (`kind: "reference"`, per-sample loop — it raises for batch > 1) and the C / OpenMP port of oracle/ is reported
  next to it under `port`; otherwise the port is the line."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  wl = make_workload(args)
  if wl.key == "builder_fixed":
    _emit(json.dumps({"impl": "reference", "unavailable": "the fixed-canvas merge has no reference implementation"}))
    return
  threads = os.cpu_count() or 1

  def measure(setup, kind):
    setup(threads)
    for _ in range(max(min(args.warmup, 3), 1)):
      wl.cpu_fn()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
      wl.cpu_fn()
    el = time.perf_counter() - t0
    return {"value": wl.cpu_units * steps / el, "unit": wl.unit, "cores": threads, "kind": kind,
            "sample": f"{wl.cpu_sample}; {steps} passes of {wl.cpu_units} units in {el:.1f} s"}, steps, el

  port, steps, el = measure(wl.cpu_setup, "port")
  line, ref_error = port, None
  if hasattr(wl, "ref_setup"):
    if reference_importable():
      try:
        line, steps, el = measure(wl.ref_setup, "reference")
      except Exception as e:  # the arm must print its line whatever happens to the optional leg
        ref_error = f"{type(e).__name__}: {e}"[:200]
    else:
      ref_error = "the reference is not importable here (no /root/reference, no baseline/_ref): the port is the line"
  out = {
    "impl": "reference", "metric": wl.metric, "value": line["value"], "unit": wl.unit, "n_gpus": args.gpus, "steps": steps,
    "warmup": max(min(args.warmup, 3), 1), "ms_per_step": 1e3 * el / steps, "higher_is_better": True, "scaling": "weak",
    "vs_baseline": None, "dtype": "f32", "data": "synthetic",
    "config": wl.config(1),
    "cpu_baseline": line,
    "e2e": {"value": line["value"], "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
  }
  if line is not port:
    out["port"] = port
  if ref_error:
    out["reference_note"] = ref_error
  _emit(json.dumps(out))


def pcie_rates(dev, barrier, gather):
  """Pinned-memory copy rates of every rank, all ranks copying at the same time: host→device alone, device→host
  alone, and both directions together (what the host-buffer entries do).  GB/s per rank."""
  n = 256 << 20
  try:
    h_in, h_out = torch.empty(n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
  except RuntimeError:
    return None
  d_in, d_out = torch.empty(n, dtype=torch.uint8, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
  s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

  def run(do_in, do_out, reps=6):
    torch.cuda.synchronize(dev)
    barrier()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    with torch.cuda.stream(s1):
      e[0].record()
      for _ in range(reps if do_in else 0):
        d_in.copy_(h_in, non_blocking=True)
      e[1].record()
    with torch.cuda.stream(s2):
      e[2].record()
      for _ in range(reps if do_out else 0):
        h_out.copy_(d_out, non_blocking=True)
      e[3].record()
    torch.cuda.synchronize(dev)
    gbs = lambda a, b_: reps * n / (a.elapsed_time(b_) * 1e-3) / 1e9
    return (gbs(e[0], e[1]) if do_in else 0.0, gbs(e[2], e[3]) if do_out else 0.0)

  run(True, True, reps=1)
  h2d, _ = run(True, False)
  _, d2h = run(False, True)
  h2d_dx, d2h_dx = run(True, True)
  rows = gather([h2d, d2h, h2d_dx, d2h_dx])
  return {"unit": "GB/s per rank, all ranks copying at once (pinned, 256 MiB x 6)",
          "h2d": [r[0] for r in rows], "d2h": [r[1] for r in rows],
          "h2d_duplex": [r[2] for r in rows], "d2h_duplex": [r[3] for r in rows]}


def time_steps(wl, steps, barrier, max_over_ranks, world):
  """`steps` steps of wl between two events on the current stream, max over ranks."""
  if hasattr(wl, "reset_counters"):
    wl.t = 0
    wl.reset_counters()
  barrier()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  trace = [] if os.environ.get("DM_BENCH_TRACE") else None
  ev0.record()
  for _ in range(steps):
    t_ = time.perf_counter()
    wl.step()
    if trace is not None:
      trace.append(time.perf_counter() - t_)
  ev1.record()
  barrier()
  if trace:  # where the host time of the timed steps went (diagnostics, stderr)
    top = sorted(range(len(trace)), key=lambda i: -trace[i])[:5]
    print(f"[trace] {type(wl).__name__}/{getattr(wl, 'key', '')}: host us/step median {1e6 * sorted(trace)[len(trace) // 2]:.0f}, "
          f"slowest {[(i, round(1e6 * trace[i])) for i in top]}", file=sys.stderr)
  ms = max_over_ranks(ev0.elapsed_time(ev1))
  algo = wl.algo_bytes_total / steps if isinstance(wl, BuilderWorkload) else wl.algo_bytes_per_step
  return ms / steps, world * wl.units_per_step * steps / (ms * 1e-3), algo


def run_extras(args, dev, rank, world, barrier, max_over_ranks, peak):
  """The other named configurations, each a short measurement of its own outside the headline region: value, ms
  per step and the roofline fraction of its step (algorithmic bytes / event time / measured HBM peak)."""
  out = {}
  shared_frames = None
  for key, steps in (("proj_labels", 100), ("flow", 100), ("builder", 100), ("builder_fixed", 100), ("proj5", 24),
                     ("proj5_labels", 24)):
    try:
      wl = make_workload(args, key)
      if isinstance(wl, BuilderWorkload):
        wl.setup(dev, rank, frames=shared_frames)
        shared_frames = wl.frames
      else:
        wl.setup(dev, rank)
      # MapBuilder: one whole episode of warm-up — the timed episode then finds the allocator's cached blocks, as every
      # episode after the first of a long-running mapping loop does
      for _ in range(wl.EPISODE if isinstance(wl, BuilderWorkload) else 3):
        wl.step()
      ms, value, algo = time_steps(wl, steps, barrier, max_over_ranks, world)
      out[key] = {"value": value, "unit": wl.unit, "ms_per_step": ms, "steps": steps,
                  "roofline_frac": algo / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_step": algo,
                  "workload": wl.config(world)["workload"]}
      if key == "builder_fixed":
        shared_frames = None
    except Exception as e:  # an extra that fails must not cost the headline line
      out[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
    wl = None
    torch.cuda.empty_cache()
  try:
    out["proj5_job"] = proj5_job(dev, rank, world, barrier, max_over_ranks)
  except Exception as e:
    out["proj5_job"] = {"error": f"{type(e).__name__}: {e}"[:300]}
  torch.cuda.empty_cache()
  return out


def run_ours(args):
  import torch.distributed as dist
  from dungeon_maps_b200 import _native as nat, shard

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if not torch.cuda.is_available():
    raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries the one JSON line and nothing else
    dist.init_process_group("nccl", device_id=dev)
    shard.bind_to_gpu_numa_node(local)  # the e2e leg streams GBs through pinned host memory per rank
  barrier = lambda: shard.barrier(dev)
  max_over_ranks = lambda x: shard.max_over_ranks(x, dev)
  sum_over_ranks = lambda x: shard.sum_over_ranks(x, dev)

  def gather(vals):  # every rank's list of floats, as rows
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    if world == 1:
      return [t.tolist()]
    rows = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(rows, t)
    return [r.tolist() for r in rows]

  wl = make_workload(args)
  if args.workload == "proj5_job":
    raise SystemExit("proj5_job is reported under `extra` of the default line (python bench.py)")
  wl.setup(dev, rank)  # every rank owns its own environments (weak scaling, no data-path collective)
  warmup = max(args.warmup, 3)
  if isinstance(wl, BuilderWorkload):
    warmup = max(warmup, wl.EPISODE)  # one whole episode: see run_extras
  for _ in range(warmup):
    wl.step()
  if hasattr(wl, "reset_counters"):
    wl.t = 0
    wl.reset_counters()
  barrier()
  sampler = ClockSampler(local) if rank == 0 else None
  if sampler:
    sampler.wait_ready()
  barrier()
  launches0 = nat.launch_count()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t_wall0 = time.perf_counter()
  ev0.record()
  for _ in range(args.steps):
    wl.step()
  ev1.record()
  barrier()
  t_wall1 = time.perf_counter()
  launches = nat.launch_count() - launches0
  ms_total = max_over_ranks(ev0.elapsed_time(ev1))
  clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
  ms_per_step = ms_total / args.steps
  value = world * wl.units_per_step * args.steps / (ms_total * 1e-3)
  total_launches = int(sum_over_ranks(float(launches)))
  algo_bytes = wl.algo_bytes_total / args.steps if isinstance(wl, BuilderWorkload) else wl.algo_bytes_per_step
  if args.dump_outputs and rank == 0:
    dump_outputs(wl.outputs(), args.dump_outputs)

  # ---- e2e: HOST buffers through the public entry, copies inside the timed region
  # cheap steps (a MapBuilder step is < 1 ms) are timed over more of them: five would be one hiccup away from noise
  e2e_steps = max(2, min(args.steps, max(args.e2e_steps, getattr(wl, "e2e_min_steps", 0))))

  def e2e_leg(**setup_kw):
    error = None
    try:  # the leg pins GBs of host memory per rank: a box that refuses must not cost the device-resident line
      wl.e2e_setup(**setup_kw)
      wl.e2e_step()
      wl.e2e_step()
    except (RuntimeError, MemoryError) as e:
      error = f"{type(e).__name__}: {e}"[:200]
    # every rank takes the same branch (a collective below): one failing rank cancels the leg for all
    if sum_over_ranks(1.0 if error else 0.0) > 0:
      error = error or "another rank could not set the host-buffer leg up"
      return {"value": None, "unit": wl.unit, "h2d_bytes_per_step": int(getattr(wl, "h2d", 0)),
              "d2h_bytes_per_step": int(getattr(wl, "d2h", 0)), "steps": 0,
              "path": getattr(wl, "e2e_path", "") + " [not measured: " + error + "]"}
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
      wl.e2e_step()
    torch.cuda.synchronize(dev)
    secs = max_over_ranks(time.perf_counter() - t0)
    wl.e2e_check()
    return {"value": world * wl.units_per_step * e2e_steps / secs, "unit": wl.unit, "h2d_bytes_per_step": int(wl.h2d),
            "d2h_bytes_per_step": int(wl.d2h), "steps": e2e_steps, "path": wl.e2e_path,
            "h2d_gbs_per_rank": wl.h2d * e2e_steps / secs / 1e9, "d2h_gbs_per_rank": wl.d2h * e2e_steps / secs / 1e9,
            "check": "outputs compared with the device-resident path / the oracle: identical"}

  skipped = {"value": None, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "steps": 0,
             "path": "not measured (--e2e-steps 0: kernel experiments)"}
  e2e = e2e_leg() if args.e2e_steps > 0 else skipped
  e2e_float32 = e2e_leg(float32=True) if (args.e2e_steps > 0 and isinstance(wl, ProjWorkload) and not wl.labels) else None
  pcie = pcie_rates(dev, barrier, gather) if args.e2e_steps > 0 else None
  peak, peak_src = measured_peak()

  extra = None
  if args.workload == "proj" and not args.no_extra:
    wl.batches, wl.depth, wl.values, wl.label_ids, wl.out, wl.last = [], None, None, None, None, None
    torch.cuda.empty_cache()
    extra = run_extras(args, dev, rank, world, barrier, max_over_ranks, peak)

  cpu = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    cpu = cpu_baseline(wl, os.cpu_count() or 1)

  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  if rank != 0:
    return
  achieved = algo_bytes / (ms_per_step * 1e-3) / 1e9
  roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
              "traffic": ncu_traffic(wl.key), "peak_source": peak_src, "algorithmic_bytes_per_step": algo_bytes,
              "kernel": wl.kernel}
  line = {
    "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": args.steps,
    "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
    "vs_baseline": None, "dtype": "f32", "data": "synthetic",
    "config": wl.config(world),
    "clocks": clocks,
    "e2e": e2e,
    "gpu_launches": total_launches,
    "roofline": roofline,
    "cpu_baseline": cpu,
  }
  if e2e_float32 is not None:
    line["e2e_float32"] = e2e_float32
  if pcie is not None:
    line["pcie"] = pcie
  if extra is not None:
    line["extra"] = extra
  _emit(json.dumps(line))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=200)
  ap.add_argument("--warmup", type=int, default=10)
  ap.add_argument("--impl", choices=("ours", "reference"), default="ours")
  ap.add_argument("--workload", choices=("proj", "flow", "builder", "builder_fixed", "proj5", "proj_labels", "proj5_labels", "proj5_job"),
                  default="proj")
  ap.add_argument("--scene", choices=("room", "iid"), default="room")
  ap.add_argument("--e2e-steps", type=int, default=5)
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-extra", action="store_true", help="skip the `extra` legs (other configs) of the default line")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help=f"write what the last timed step returned as DIR/<name>.npy (float32 / float64, at most "
                       f"{DUMP_BYTES >> 20} MiB in all: larger outputs as a fixed seeded sample of their elements)")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl != "ours":
    ap.error("--dump-outputs writes the outputs of --impl ours")
  if args.gpus > 1 and args.impl == "ours" and "WORLD_SIZE" not in os.environ:
    # called directly with --gpus N: become the torchrun launch the driver would have made (one rank per GPU)
    import socket
    with socket.socket() as sock:
      sock.bind(("127.0.0.1", 0))
      port = sock.getsockname()[1]
    os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                              f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1", "--master-port", str(port),
                              os.path.abspath(__file__)] + sys.argv[1:])
  # stdout carries the one JSON line and nothing else: libraries that print from C (NCCL's version banner ignores
  # NCCL_DEBUG_FILE on some boxes) get stderr as their fd 1 while the run lasts
  sys.stdout.flush()
  real_stdout = os.dup(1)
  os.dup2(2, 1)
  try:
    if args.impl == "reference":
      run_reference(args)
    else:
      run_ours(args)
  finally:
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    os.close(real_stdout)
  if _RESULT_LINE:
    print(_RESULT_LINE[0], flush=True)


if __name__ == "__main__":
  main()
