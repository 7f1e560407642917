/*
 * dungeon_maps_b200 — C ABI of the B200-native depth → top-down hot path.
 *
 * Every entry point below is what the reference's Python layer would bind
 * (ctypes) in place of the body of one of its own functions.  The reference
 * interface each one replaces is cited as /root/reference file:line.
 *
 * Conventions
 *   - plain pointers + sizes only, no torch types; all `const float*` etc. are
 *     DEVICE pointers unless the function name ends in `_host`.
 *   - all tensors are dense, C-contiguous, float32 / uint8 (bool) / int64.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - return value: 0 on success, a positive cudaError_t value on a CUDA
 *     failure, a negative DM_E* code on a usage error.  Nothing is printed.
 *   - arithmetic follows the reference's float32 op order exactly (one IEEE
 *     rounding per torch op, FMA only where the reference's sgemm used it);
 *     see DESIGN.md "Numerics".
 */
#ifndef DUNGEON_MAPS_B200_H_
#define DUNGEON_MAPS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DM_ABI_VERSION 3

#define DM_OK 0
#define DM_EINVAL (-1)     /* bad argument (null pointer, non-positive size, ...) */
#define DM_EWORKSPACE (-2) /* workspace too small */
#define DM_ETIMEOUT (-3)   /* device-side dependency wait timed out (bug guard) */

/* One rigid step of the reference's space transforms.
 *   kind 1 (ROT_THEN_ADD): p' = rot(R, p) + t      camera_to_local_space  maps.py:753-800
 *                                                  local_to_global_space  maps.py:850-895
 *   kind 2 (ADD_THEN_ROT): p' = rot(R, p + t)      local_to_camera_space  maps.py:802-848
 *                                                  global_to_local_space  maps.py:897-942
 *   kind 3 (ADD): p' = p + t                        utils.translate        utils.py:229-259
 *   kind 4 (ROT): p' = rot(R, p)                    utils.rotate           utils.py:261-330
 *   kind 0: identity (step skipped)
 * rot(R, p)_i, utils.py:329 (einsum 'bji,b...j->b...i' → at::bmm), depends on how many
 * points n the reference rotates in one call, because ATen switches kernels:
 *   fused = 1 (9*n >= 400, MKL sgemm):   fma(R[2][i], p2, fma(R[1][i], p1, R[0][i]*p0))
 *   fused = 0 (9*n <  400, naive loop):  (R[0][i]*p0 + R[1][i]*p1) + R[2][i]*p2, each op rounded
 * R is the Rodrigues matrix built on the host exactly as utils.py:303-327 does.
 */
#define DM_STEP_NONE 0
#define DM_STEP_ROT_THEN_ADD 1
#define DM_STEP_ADD_THEN_ROT 2
#define DM_STEP_ADD 3
#define DM_STEP_ROT 4

typedef struct DmStep {
  float R[9]; /* row-major R[j][i] = R[3*j+i] */
  float t[3];
  int32_t kind;
  int32_t fused;
  int32_t _pad[2];
} DmStep; /* 64 bytes */

/* Per-sample parameters of orth_project (maps.py:127-351). */
typedef struct DmProjSample {
  DmStep to_local;  /* pitch about x, + (0, cam_height, 0) */
  DmStep to_global; /* yaw about y, + (x, 0, z); kind 0 when to_global is False */
  float width_offset;
  float height_offset;
  float _pad[14];
} DmProjSample; /* 192 bytes */

/* Batch-wide configuration of orth_project. */
typedef struct DmProjCfg {
  int32_t H, W;      /* depth frame */
  int32_t C;         /* value channels; 0: the heights are the values (value_map None) */
  int32_t Mh, Mw;    /* map_height, map_width */
  float fx, fy, cx, cy;
  float map_res;
  float trunc_depth_min, trunc_depth_max, trunc_height_max;
  int32_t has_trunc_depth_min, has_trunc_depth_max, has_trunc_height_max;
  int32_t clip_border;
  int32_t flip_h;
  float fill_value;  /* effective initial canvas value: fill_value, or 0 when None (utils.py:472-473) */
  int32_t want_height; /* C>0 only: also produce the 1-channel height map (maps.py:335-349) */
  int32_t reduction;   /* 0 = max (Reduction.max / None), 1 = min */
  int32_t fast_steps;  /* caller's promise about EVERY sample, enabling straight-line transform code:
                          0: nothing promised (steps are interpreted per sample);
                          1: to_local is {ROT_THEN_ADD, fused, R a rotation about x: R[0]=1,
                             R[1]=R[2]=R[3]=R[6]=0, t=(0,h,0)} and to_global is NONE;
                          2: as 1, and to_global is {ROT_THEN_ADD, fused, R a rotation about y:
                             R[4]=1, R[1]=R[3]=R[5]=R[7]=0, t=(x,0,z)}.
                          Multiplications by those exact 0/1 entries are skipped; results are
                          identical for every pixel that lands on the map (DESIGN.md "Numerics"). */
  int32_t _pad[3];
} DmProjCfg;

/* Fused orthographic projection.  Replaces the body of orth_project
 * (maps.py:259-351): depth_map_to_point_cloud, _mask_borders,
 * camera_to_local_space, height truncation, local_to_global_space,
 * map_quantize, project/scatter_tensor (utils.py:389-492) and the second
 * height scatter — without materialising the point cloud.
 *
 *   depth   (b, 1, H, W) f32
 *   values  (b, C, H, W) f32 or NULL when cfg->C == 0
 *   valid   (b, 1, H, W) u8  or NULL
 *   samples b entries
 *   topdown (b, max(C,1), Mh, Mw) f32   out
 *   mask    (b, max(C,1), Mh, Mw) u8    out   "cell changed" mask (utils.py:489-491)
 *   height  (b, 1, Mh, Mw) f32          out, may be NULL unless cfg->want_height
 *   workspace: device scratch of at least dm_orth_project_workspace_bytes();
 *     it must be zero-filled before its first use and may be reused across
 *     calls (every call leaves it zero-filled again).
 */
size_t dm_orth_project_workspace_bytes(const DmProjCfg* cfg, int32_t b);
int dm_orth_project_f32(const float* depth, const float* values, const uint8_t* valid,
                        const DmProjSample* samples, const DmProjCfg* cfg, int32_t b,
                        float* topdown, uint8_t* mask, float* height,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Same call with HOST buffers: copies inputs host→device, runs
 * dm_orth_project_f32, copies the outputs back.  `samples` and `cfg` are host
 * structs in both variants' cfg; here `samples` is a host array too.  Device
 * scratch is owned by the library (grown on demand, released by
 * dm_release_scratch).  Pinned host memory makes the copies asynchronous. */
int dm_orth_project_host_f32(const float* depth, const float* values, const uint8_t* valid,
                             const DmProjSample* samples, const DmProjCfg* cfg, int32_t b,
                             float* topdown, uint8_t* mask, float* height, int32_t device);
void dm_release_scratch(void);

/* Class-id form of the projection, for the reference's semantic usage: demos/object_map/run.py:117-124 feeds
 * orth_project with value_map = one_hot(segmentation, num_classes).float().  This entry takes the ids themselves,
 *   labels (b, 1, H, W) u8, cfg->C = num_classes (1..63),
 * and writes exactly (bit for bit) what dm_orth_project_f32 writes for values[b][c][p] = (labels[b][p] == c) ? 1 : 0
 * (an id >= num_classes is an all-zero row): same outputs, same mask rule, same fill_value / reduction (max, min) /
 * want_height semantics, any H, W and alignment.  A pixel costs 5 input bytes instead of 4 * (C + 1) and a run of
 * pixels in one cell two atomic reductions (height key, class-presence word) instead of C + 1.
 * The workspace follows the rules of dm_orth_project_f32 (zero before first use, left zeroed) and may be the same
 * buffer, provided it is large enough for both. */
size_t dm_orth_project_labels_workspace_bytes(const DmProjCfg* cfg, int32_t b);
int dm_orth_project_labels_f32(const float* depth, const uint8_t* labels, const uint8_t* valid,
                               const DmProjSample* samples, const DmProjCfg* cfg, int32_t b,
                               float* topdown, uint8_t* mask, float* height,
                               void* workspace, size_t workspace_bytes, void* stream);
/* HOST-buffer variant (see dm_orth_project_host_f32): 5 bytes per pixel cross PCIe instead of 4 * (C + 1). */
int dm_orth_project_labels_host_f32(const float* depth, const uint8_t* labels, const uint8_t* valid,
                                    const DmProjSample* samples, const DmProjCfg* cfg, int32_t b,
                                    float* topdown, uint8_t* mask, float* height, int32_t device);

/* Uploads a small host-built parameter block (per-sample transforms, fuse sources, ...; at most 64 KiB) for the NEXT
 * call queued on `stream` of the current device: copied through the library's ring of pinned slots on a copy stream of
 * its own, `stream` waits for the copy.  *dev_ptr stays valid for the work queued on `stream` before the 64th upload
 * after this one.  (What the Python layer used torch for: pinned staging + copy on the caller's stream, which put a
 * copy-engine round trip between the kernels of consecutive calls.) */
int dm_upload_params(const void* src, size_t nbytes, void* stream, void** dev_ptr);

/* Device-side wait guard.  The projection kernels are persistent launches whose CTAs wait on one another's
 * per-frame completion counters; a wait that exceeds 4 s (a scheduling bug, never expected) does not hang the GPU:
 * the item is skipped, the launch re-zeroes its workspace before it ends, and DM_ETIMEOUT is reported ONCE by
 * whichever comes first of: the next dm_orth_project*_f32 call on that device (which then launches nothing), the
 * final synchronisation of a *_host entry, or dm_device_status(device) (reads and clears the flag; call it after
 * synchronising the stream).  The outputs of the timed-out call are undefined. */
int dm_device_status(int32_t device);
/* Test hook: spin_ns = guard time of the waits (0: the 4 s default); dep_bias is added to every dependency target
 * (non-zero: no dependency is ever satisfied, every dependent item times out). */
void dm_debug_set_wait_guard(uint64_t spin_ns, uint32_t dep_bias);
/* Test hook: frames per chunk of the *_host entries' copy / kernel / copy pipeline (0: chosen from the frame size). */
void dm_debug_set_host_chunk(int32_t frames);
/* Tile layout of the float projection kernel. -1: automatic (the fastest measured layout: tiles of 512 consecutive
 * pixels staged by bulk copies), 0: the same, forced, 4 / 8: 2-D tiles of that many image rows x 128 / 64 columns staged
 * by one tensor-map TMA copy per tile (cp.async.bulk.tensor.3d; folds vertical runs before they leave the SM — fewer
 * REDs, more instructions: slower on the B200, DESIGN.md §3).  Every layout produces the same bits. */
void dm_debug_set_tile_rows(int32_t rows);
/* Test hook: 0 keeps the merge's first source on the per-cell scatter for every plane; 1 (default) lets planes whose
 * cells all move by one whole (dx, dz) be copied densely (dm_fuse.cu: plane_shift).  Same bits either way. */
void dm_debug_set_dense_shift(int32_t on);

/* Per-sample parameters of camera_affine_grid (maps.py:353-460). */
typedef struct DmFlowSample {
  DmStep to_local;   /* pitch, +cam_height                    maps.py:428-433 */
  DmStep transition; /* yaw delta about y, + (dx, 0, dz)      maps.py:435-439 */
  DmStep to_camera;  /* + (0,-cam_height,0) then rot(-pitch)  maps.py:441-446 */
} DmFlowSample; /* 192 bytes */

typedef struct DmFlowCfg {
  int32_t H, W;
  int32_t channels; /* depth channels per sample (grid is (b, channels, H, W, 2)) */
  float fx, fy, cx, cy;
  int32_t flip_h;
  int32_t emit_flow; /* 0: grid (camera_affine_grid). 1: ego flow of the demo helper
                        compute_ego_flow (demos/ego_flow/run.py:75-90):
                        (x - gx, -(y - gy)) */
  int32_t _pad[6];
} DmFlowCfg;

/* Fused unproject → transform → reproject.  Replaces the body of
 * camera_affine_grid (maps.py:414-460).
 *   depth (b, channels, H, W) f32 ; grid (b, channels, H, W, 2) f32 out */
int dm_affine_grid_f32(const float* depth, const DmFlowSample* samples, const DmFlowCfg* cfg,
                       int32_t b, float* grid, void* stream);

/* ---- MapBuilder merge: fuse_topdown_maps (maps.py:2181-2287) ---------------- */

/* One source map of a fusion, all samples sharing its geometry.  The DmFuseSource array
 * handed to the two calls below lives in HOST memory (at most 8 sources per call); the
 * pointers inside it are device pointers. */
typedef struct DmFuseSource {
  const float* height;   /* (b, C, h, w) f32; channel stride may be 0 (stride-0 expand, maps.py:349) */
  const float* values;   /* (b, C, h, w) f32 or NULL for a height map */
  const uint8_t* mask;   /* (b, C, h, w) u8 */
  int64_t height_bstride, height_cstride; /* in elements */
  int32_t h, w;          /* this map's map_height, map_width */
  int32_t flip_h;
  float map_res;
  const float* width_offset;  /* (b,) device */
  const float* height_offset; /* (b,) device */
  const DmStep* steps;   /* (b, 2) device: [source local→global or none, global→target local or none]
                            _flattened_topdown_map maps.py:2059-2060, _merge_point_clouds maps.py:2116-2117 */
  const int32_t* plane_box; /* optional, (b*C, 4) int32 device, 16-byte aligned: per plane the rows [min, max] and
                            columns [min, max] that hold all of its valid cells, as dm_fuse_scatter_track_f32 left
                            them for a map it wrote (max < min: the plane has no valid cell).  The passes then scan
                            that rectangle instead of the whole plane.  NULL: scan everything. */
} DmFuseSource;

/* Pass 1: bounding box of every valid point of every source in bins of the
 * target resolution with zero offsets and no flip
 * (_compute_new_shape_and_offsets, maps.py:2146-2179).
 * out (device, 5×int64): min_x, max_x, min_z, max_z, n_valid.  The caller
 * initialises nothing; the call overwrites all five. */
int dm_fuse_bbox_i64(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                     float target_res, int64_t* out, void* stream);
/* The same, starting from `seed` (device, 5×int64, may be NULL) instead of an empty box: the bounding box that
 * dm_fuse_scatter_track_f32 left for a map that would otherwise be one of the sources.  A MapBuilder's world map is
 * by far the largest source of every merge (maps.py:2471-2508) and its contribution to the box is a function of
 * the map alone, so it is reduced once, while the map is written, instead of by a scan before every host sync.
 * n_sources may be 0 when seed is given. */
int dm_fuse_bbox_seeded_i64(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                            float target_res, const int64_t* seed, int64_t* out, void* stream);

/* Pass 2: re-quantise every valid point with the new offsets and scatter-max
 * it into the freshly sized canvases (maps.py:2232-2272).
 *   topdown (b, C, Mh, Mw) f32 out; mask (b, C, Mh, Mw) u8 out;
 *   height  (b, C, Mh, Mw) f32 out, NULL for height maps (then topdown is the height map). */
typedef struct DmFuseTarget {
  int32_t Mh, Mw;
  int32_t flip_h;
  float map_res;
  float width_offset, height_offset; /* scalars: one bbox over the whole batch */
  float fill_value;
  int32_t reduction;
} DmFuseTarget;
int dm_fuse_scatter_f32(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                        const DmFuseTarget* target, float* topdown, uint8_t* mask, float* height,
                        void* stream);
/* The same, and next_bbox (device, 5×int64, overwritten; may be NULL) receives what dm_fuse_bbox_i64 would compute
 * for the map written here when it is later passed as a global-frame source (identity steps) with the same
 * map_res, offsets and flip_h as `target`: min_x, max_x, min_z, max_z over its valid cells, and a count that is
 * zero iff the map has no valid cell (NOT the number of valid cells).  DM_EINVAL with a NaN fill_value. */
/* next_plane_box (device, (b*C, 4) int32, overwritten; may be NULL): per plane of the map written here, the rows and
 * columns that hold its valid cells — DmFuseSource.plane_box of a later merge. */
int dm_fuse_scatter_track_f32(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                              const DmFuseTarget* target, float* topdown, uint8_t* mask, float* height,
                              int64_t* next_bbox, int32_t* next_plane_box, void* stream);

/* Opt-in fixed-canvas merge (SURVEY.md §8f-2; no reference call does this — the closest is
 * project(..., canvas=, canvas_masks=), maps.py:1089-1173 with utils.py:462-491, whose semantics it keeps):
 * the valid cells of the sources are re-projected and max/min-merged IN PLACE into canvases that
 * already hold a world map; mask |= "cell now differs from fill_value".  One launch, no host sync.
 * target->width_offset/height_offset are the canvases' fixed offsets. */
int dm_fuse_inplace_f32(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                        const DmFuseTarget* target, float* topdown, uint8_t* mask, float* height,
                        void* stream);
/* Fresh canvases for the call above: topdown = fill_value, height = -inf (NULL for height maps), mask = 0;
 * n = b*C*Mh*Mw cells. */
int dm_fuse_canvas_init_f32(float* topdown, uint8_t* mask, float* height, int64_t n, float fill_value,
                            void* stream);
/* Clears the samples of a batched map that are done (MapBuilder.reset_envs), in place, on the device:
 *   topdown (b, C, Mh, Mw) f32, height (b, C, Mh, Mw) f32 (NULL for height maps), mask (b, C, Mh, Mw) u8;
 *   done (b,) u8 device, read by the kernels only: every plane of a sample with done[s] != 0 gets fill_value / -inf / 0,
 *   whole; the other planes are not touched.
 *   map: Mh, Mw, flip_h, map_res, width_offset, height_offset, fill_value and reduction of the map.
 *   plane_box (optional, (b*C, 4) int32 device, 16-byte aligned, as dm_fuse_scatter_track_f32 left it): the cleared
 *   planes' rectangles become empty (max < min), the others stay.
 *   box (optional, 5 x int64 device; requires plane_box): rebuilt from the surviving rectangles, what
 *   dm_fuse_bbox_i64 finds for the cleared map; its count is the number of non-empty planes (zero iff no valid cell).
 *   With no sample done, plane_box and box are left as they are.
 * DM_EINVAL for null tensors, b <= 0, C <= 0, a box without plane_box, and a box or plane_box with a NaN fill_value or
 * reduction >= 2.  No host synchronisation, no copy. */
int dm_fuse_clear_envs_f32(float* topdown, float* height, uint8_t* mask, int32_t b, int32_t C, const uint8_t* done,
                           const DmFuseTarget* map, int32_t* plane_box, int64_t* box, void* stream);

/* ---- per-sample parameter blocks packed on the host, in C ------------------------------------------------------
 * What the kernels need per sample derives from a pose (x, z, yaw) and per-call constants.  These two functions are
 * pure host code (no device work, no sin / cos): the caller supplies sin(yaw) / cos(yaw) of the raw yaw computed with
 * the reference's own torch-CPU ops (utils.py:325-326; the |a| <= 0.001 → 0 clamp of utils.py:323-324 is applied
 * here: sin = 0, cos = 1), and the yaw rotation is formed as (I + sin S) + (1 - cos) S² in float32, the reference's
 * operation order (utils.py:318-327). */
typedef struct DmPoseCfg {
  float pitch_R[9];      /* camera_to_local_space: rotation about x by cam_pitch (maps.py:789-793), host-built */
  float pitch_back_R[9]; /* local_to_camera_space: rotation about x by -cam_pitch (maps.py:838-842); flow only */
  float cam_height;
  float yaw_skew[9], yaw_skew_sq[9]; /* S and S² of the axis (0, 1, 0) as utils.py:303-318 builds them */
  int32_t fused;         /* DmStep.fused of every step: 9 * (points rotated per sample) >= 400 */
  int32_t _pad[2];
} DmPoseCfg;
/* orth_project (maps.py:279-295): to_local = rot(pitch) + (0, h, 0); to_global = rot(yaw) + (x, 0, z), or none.
 * pose (b, 3), sin_yaw / cos_yaw (b,) may be NULL unless to_global; width_offset / height_offset (b,).
 * *fast_steps receives the DmProjCfg.fast_steps value these blocks allow. */
int dm_pack_proj_samples(const DmPoseCfg* cfg, const float* pose, const float* sin_yaw, const float* cos_yaw,
                         const float* width_offset, const float* height_offset, int32_t to_global, int32_t b,
                         DmProjSample* out, int32_t* fast_steps);
/* camera_affine_grid (maps.py:428-446): to_local, transition by trans_pose, to_camera. */
int dm_pack_flow_samples(const DmPoseCfg* cfg, const float* pose, const float* sin_yaw, const float* cos_yaw,
                         int32_t b, DmFlowSample* out);
/* TopdownMap.select_egocentric: DM_EGO_SAMPLE_WORDS floats per sample, out (b * DM_EGO_SAMPLE_WORDS):
 *   words 0-15  DmStep local_to_global_space(pose) = rot(yaw) + (x, 0, z);
 *   words 16-17 the source map's width / height offsets;
 *   words 18-19 the window's width / height offsets.
 * Only cfg->yaw_skew, yaw_skew_sq and fused are read; fused = 9 * crop_h * crop_w >= 400 (the window's cells are the
 * points the composition rotates per sample).  All arrays (b,) except pose (b, 3). */
#define DM_EGO_SAMPLE_WORDS 20
int dm_pack_ego_samples(const DmPoseCfg* cfg, const float* pose, const float* sin_yaw, const float* cos_yaw,
                        const float* src_width_offset, const float* src_height_offset, const float* width_offset,
                        const float* height_offset, int32_t b, float* out);

/* ---- MapBuilder.step with the host side in C (maps.py:2357-2508) ----------------------------------------------
 * The plot → merge loop of b environments for height maps (value_map None) and a world map in the global frame —
 * the configuration a mapping loop runs thousands of times.  A step packs every parameter block (projection
 * samples, the fuse sources of world and local map) into one pinned slot, uploads it with one copy and launches the
 * kernels back to back; the caller allocates the map tensors.  Results are those of dm_orth_project_f32 +
 * dm_fuse_bbox_seeded_i64 + dm_fuse_scatter_track_f32 called one by one (the functions used inside). */
typedef struct DmBuilder DmBuilder; /* opaque */

typedef struct DmBuilderCfg {
  DmProjCfg proj;          /* projection of the local maps (maps.py:2447-2458); C: 0 for dm_builder_create, the
                              channel count for dm_builder_create_values; fast_steps, want_height are derived */
  int32_t b;               /* environments */
  int32_t plot_to_global;  /* the local maps are plotted in the global frame (to_global of the plot call) */
  float pitch_R[9];        /* DmStep.R of camera_to_local_space: rotation about x by cam_pitch, built on the host by
                              the reference's own ops (utils.py:303-327) */
  float cam_height;
  float width_offset, height_offset; /* of the local maps */
  float yaw_skew[9], yaw_skew_sq[9]; /* S and S² of the axis (0, 1, 0) as utils.py:303-318 builds them: the yaw
                              rotation of a step is (I + sin S) + (1 - cos) S², float32, in that order */
  float merge_fill_value;  /* fill_value of the merged canvases (maps.py:2246-2254) */
  int32_t merge_reduction; /* 0 max, 1 min */
  int32_t _pad[2];
} DmBuilderCfg;

/* A (b, 1, h, w) height map in the global frame, tensors on the device. */
typedef struct DmMapRef {
  float* topdown;
  uint8_t* mask;
  int32_t h, w;
  float width_offset, height_offset;
  int64_t* box; /* device, 5 x int64: as a source, the box dm_fuse_scatter_track_f32 left for this map (NULL: scan
                   it); as the output of dm_builder_merge, where that box is written (NULL: not tracked) */
  int32_t* plane_box; /* device, (b, 4) int32: the per-plane rectangles of valid cells, same roles (NULL: none) */
} DmMapRef;

/* Size and offsets of the canvas the merge needs (_compute_new_shape_and_offsets, maps.py:2146-2179). */
typedef struct DmMergeShape {
  int64_t n_valid; /* 0: no valid point anywhere, the merge is skipped (maps.py:2217-2225) */
  int32_t map_height, map_width;
  float width_offset, height_offset;
} DmMergeShape;

int dm_builder_create(const DmBuilderCfg* cfg, int32_t device, DmBuilder** out);
void dm_builder_destroy(DmBuilder* builder);
/* Step, first half: plots the local maps of `depth` (b, 1, H, W) at `pose` (HOST, (b, 3) = x, z, yaw; sin_yaw /
 * cos_yaw: HOST (b,), of the raw yaw: the |a| <= 0.001 clamp of utils.py:323-324 is applied inside) into local_topdown / local_mask
 * (b, 1, Mh, Mw), reduces the bounding box of world ∪ local and BLOCKS until it is on the host (the reference's
 * .item() sync): `shape` says what to allocate.  world may be NULL (empty world map). */
int dm_builder_plot(DmBuilder* builder, const float* depth, const float* pose, const float* sin_yaw,
                    const float* cos_yaw, float* local_topdown, uint8_t* local_mask, const DmMapRef* world,
                    DmMergeShape* shape, void* stream);
/* dm_builder_plot with speculation: prefill_topdown / prefill_mask (prefill_cells elements each; may be NULL / 0) are
 * canvases the caller expects to merge into — as a rule the size class of the old world map.  Their fill is queued right
 * behind the bounding box's copy and runs while the host waits for the box; dm_builder_merge then only fills the cells of
 * `out` beyond prefill_cells (rounded down to a multiple of 16) when `out` points at them.  Same results as
 * dm_builder_plot + dm_builder_merge. */
int dm_builder_plot_prefill(DmBuilder* builder, const float* depth, const float* pose, const float* sin_yaw,
                            const float* cos_yaw, float* local_topdown, uint8_t* local_mask, const DmMapRef* world,
                            DmMergeShape* shape, float* prefill_topdown, uint8_t* prefill_mask, int64_t prefill_cells,
                            void* stream);
/* shape may be NULL in dm_builder_plot_prefill: the call then only queues its work and dm_builder_plot_wait blocks
 * for the bounding box later (the caller has ~100 us of GPU work to prepare its own bookkeeping behind). */
int dm_builder_plot_wait(DmBuilder* builder, DmMergeShape* shape);
/* Step, second half: fills `out` (shape->map_height x map_width, offsets from `shape`) and scatters the world map
 * and the local map of the preceding dm_builder_plot into it. */
int dm_builder_merge(DmBuilder* builder, const DmMapRef* out, void* stream);
/* Opt-in fixed-canvas step (dm_fuse_inplace_f32 semantics): plot, then merge in place into `canvas`; no host sync. */
int dm_builder_step_fixed(DmBuilder* builder, const float* depth, const float* pose, const float* sin_yaw,
                          const float* cos_yaw, float* local_topdown, uint8_t* local_mask, const DmMapRef* canvas,
                          void* stream);

/* The same step for value maps: MapBuilder.step(value_map=) with float planes, or step(label_map=, num_classes=) with
 * class ids (the one_hot planes of the reference's object-map loop, never materialised).  World maps carry C height
 * planes of their own (maps.py:2258-2271); the local map has one, shared by its C channels (maps.py:349).  Results are
 * those of dm_orth_project_f32 / dm_orth_project_labels_f32 (want_height) + dm_fuse_bbox_seeded_i64 +
 * dm_fuse_scatter_track_f32 / dm_fuse_inplace_f32 called one by one. */
typedef struct DmValueMapRef {
  float* topdown;     /* (b, C, h, w) f32 values */
  float* height;      /* (b, C, h, w) f32 height planes */
  uint8_t* mask;      /* (b, C, h, w) u8 */
  int32_t h, w;
  float width_offset, height_offset;
  int64_t* box;       /* as DmMapRef.box */
  int32_t* plane_box; /* device, (b * C, 4) int32: as DmMapRef.plane_box, one rectangle per (sample, channel) */
} DmValueMapRef;

/* cfg->proj.C = C channels: 1..63 with labels != 0 (class ids), >= 1 otherwise (float planes).  Reductions max / min
 * (proj.reduction and merge_reduction).  DM_EINVAL for anything else, before any CUDA call.  The handle owns the
 * workspace of the projection entry it uses.  Destroy with dm_builder_destroy. */
int dm_builder_create_values(const DmBuilderCfg* cfg, int32_t labels, int32_t device, DmBuilder** out);
/* dm_builder_plot_prefill for value maps.  Input: values (b, C, H, W) f32 (labels NULL) or labels (b, 1, H, W) u8
 * (values NULL), as the handle was created.  Output: local_topdown / local_mask (b, C, Mh, Mw), local_height
 * (b, 1, Mh, Mw).  world may be NULL.  The prefill covers three canvases of prefill_cells elements each:
 * prefill_topdown = fill, prefill_height = -inf, prefill_mask = 0.  shape NULL: wait with dm_builder_plot_wait. */
int dm_builder_plot_values(DmBuilder* builder, const float* depth, const float* values, const uint8_t* labels,
                           const float* pose, const float* sin_yaw, const float* cos_yaw, float* local_topdown,
                           uint8_t* local_mask, float* local_height, const DmValueMapRef* world, DmMergeShape* shape,
                           float* prefill_topdown, float* prefill_height, uint8_t* prefill_mask, int64_t prefill_cells,
                           void* stream);
/* dm_builder_merge for value maps: fills `out` (the tail beyond a prefill) and scatters the world map and the local map
 * of the preceding dm_builder_plot_values into it; out->box / out->plane_box (may be NULL) receive the tracked boxes. */
int dm_builder_merge_values(DmBuilder* builder, const DmValueMapRef* out, void* stream);
/* dm_builder_step_fixed for value maps: plot, then merge in place into the (b, C, Hc, Wc) canvases and their height
 * planes; no host sync. */
int dm_builder_step_fixed_values(DmBuilder* builder, const float* depth, const float* values, const uint8_t* labels,
                                 const float* pose, const float* sin_yaw, const float* cos_yaw, float* local_topdown,
                                 uint8_t* local_mask, float* local_height, const DmValueMapRef* canvas, void* stream);

/* ---- materialising primitives (the reference's public L0/L1 functions) ------ */

/* points (b, n, 3) f32 → out (b, n, 3): applies steps[b][n_steps] in order.
 * utils.rotate utils.py:261-330, utils.translate utils.py:229-259 and the four
 * space transforms maps.py:753-942. */
int dm_transform_points_f32(const float* points, const DmStep* steps, int32_t n_steps,
                            int32_t b, int64_t n, float* out, void* stream);

/* image_to_camera_space maps.py:616-682 (to_image = 0) and
 * camera_to_image_space maps.py:684-751 (to_image = 1) on (n, 3) points. */
int dm_image_camera_f32(const float* points, int64_t n, float fx, float fy, float cx, float cy,
                        int32_t flip_h, int32_t height, int32_t to_image, float* out, void* stream);

/* depth_map_to_point_cloud maps.py:462-545: depth (b*c, H, W) → points (b*c, H, W, 3) and
 * valid (b*c, H, W) u8. valid_in may be NULL.  DM_EINVAL for a frame of 2^31 pixels or more. */
int dm_depth_to_points_f32(const float* depth, const uint8_t* valid_in, int64_t frames, int32_t H,
                           int32_t W, float fx, float fy, float cx, float cy, int32_t flip_h,
                           int32_t has_tmin, float tmin, int32_t has_tmax, float tmax,
                           float* points, uint8_t* valid_out, void* stream);

/* map_quantize maps.py:944-1019: x, z (b, n) f32 + offsets (b,) → bins (b, n) int64. */
int dm_map_quantize_f32(const float* x, const float* z, const float* width_offset,
                        const float* height_offset, int32_t b, int64_t n, float map_res,
                        int32_t map_height, int32_t flip_h, int64_t* x_bin, int64_t* z_bin,
                        void* stream);
/* map_dequantize maps.py:1021-1087. */
int dm_map_dequantize_f32(const float* x_bin, const float* z_bin, const float* width_offset,
                          const float* height_offset, int32_t b, int64_t n, float map_res,
                          int32_t map_height, int32_t flip_h, float* x, float* z, void* stream);

/* scatter_tensor utils.py:389-492 / project maps.py:1089-1173 for 2-D canvases:
 * values (B, N) f32, coords (B, N, 2) int64 [row, col], valid (B, N) u8 or NULL,
 * canvas_in (B, Mh, Mw) f32 (ignored / may be NULL when has_fill), canvas_out (B, Mh, Mw) f32,
 * mask (B, Mh, Mw) u8 out ("changed" vs the starting canvas).
 * reduction (utils.py:44-76): 0 max, 1 min, 2 sum, 3 mean, 4 prod.  max / min are exact; sum / mean / prod use float
 * atomics (hit order differs from the reference's index order: equal to rounding).  mean follows torch_scatter:
 * (starting canvas + sum of hits) / max(number of hits, 1). */
int dm_scatter_f32(const float* values, const int64_t* coords, const uint8_t* valid, int64_t B,
                   int64_t N, int32_t Mh, int32_t Mw, int32_t has_fill, float fill_value,
                   int32_t reduction, const float* canvas_in, float* canvas_out, uint8_t* mask,
                   void* stream);

/* crop_topdown_map maps.py:1959-2037 = generate_crop_grid utils.py:571-611 +
 * image_sample utils.py:613-652 (pad 1, grid_sample nearest, align_corners).
 * image (b, c, h, w) f32 → out (b, c, crop_h, crop_w); center (b, 2) f32 device.
 * border = 1: padding_mode 'border' with pad value `fill` (fill_value given);
 * border = 0: zeros.  DM_EINVAL for a crop or an image plane of 2^31 cells or more. */
int dm_crop_nearest_f32(const float* image, const float* center, int32_t b, int32_t c, int32_t h,
                        int32_t w, int32_t crop_h, int32_t crop_w, int32_t border, float fill,
                        float* out, void* stream);
int dm_crop_nearest_u8(const uint8_t* image, const float* center, int32_t b, int32_t c, int32_t h,
                       int32_t w, int32_t crop_h, int32_t crop_w, uint8_t* out, void* stream);

/* TopdownMap.select_egocentric: a crop_h x crop_w window of a global-frame map per sample, in the sample's camera
 * frame (not in the reference; defined by its public functions).  Output cell (r, c) of sample s:
 *   (lx, lz) = map_dequantize(c, r, window offsets, map_res, crop_h, flip_h)
 *   (gx, gz) = local_to_global_space((lx, 0, lz), pose)      (the DmStep of the sample block)
 *   (X, Z)   = map_quantize(gx, gz, source offsets, map_res, Hs, flip_h)
 *   out = source[s, k, Z, X] inside the source, else fill_value / -inf (height) / 0 (mask).
 * Source: topdown (b, C, Hs, Ws) f32, mask (b, C, Hs, Ws) u8, height f32 (NULL for height maps) with
 * height_plane_stride Hs * Ws ((b, C, Hs, Ws)) or 0 ((b, 1, Hs, Ws) shared by the C channels).
 * samples: device, b * DM_EGO_SAMPLE_WORDS floats from dm_pack_ego_samples.
 * Output: out_topdown / out_mask (b, C, crop_h, crop_w), out_height (b, C or 1, crop_h, crop_w) as the source's
 * heights, NULL exactly when height is NULL.  One launch, no host synchronisation.
 * DM_EINVAL, before any CUDA call, for null tensors, b, C, Hs, Ws, crop_h or crop_w <= 0, map_res not > 0, a window or
 * source plane of 2^31 cells or more, height and out_height not both given or both NULL, another plane stride, and
 * unaligned samples. */
int dm_crop_egocentric_f32(const float* topdown, const float* height, int64_t height_plane_stride, const uint8_t* mask,
                           int32_t b, int32_t C, int32_t Hs, int32_t Ws, float map_res, int32_t flip_h,
                           const float* samples, int32_t crop_h, int32_t crop_w, float fill_value, float* out_topdown,
                           float* out_height, uint8_t* out_mask, void* stream);

/* geodesic_distance: per-environment shortest-path distances over an 8-connected grid (not in the reference).
 * traversable (b, H, W) u8 0 / 1; the sources are EITHER source_mask (b, H, W) u8 (source_cells NULL, n_cells 0) OR
 * source_cells (b, n_cells, 2) int64 [x, z] = [column, row] (source_mask NULL, n_cells >= 1; cells outside the map are
 * ignored).  An edge runs from u to an 8-neighbour v when v is traversable and, for a diagonal step, both cells that
 * share an edge with u and with v are traversable (no corner cutting); an orthogonal step costs 5, a diagonal one 7.
 * Edges depend on the destination only: a source that is an obstacle still reaches its free neighbours.
 * dist (b, H, W) int32: 0 on sources, else the least path cost from any source of the environment, -1 without a path.
 * Exact (integer costs), whatever the evaluation order.  One cooperative launch, no host synchronisation; the kernel
 * stops after H * W + 2 rounds, a count it provably never needs, and then raises the status word dm_device_status
 * reports as DM_ETIMEOUT (dist is undefined).  DM_EINVAL, before any CUDA call, for null traversable or dist, b, H or
 * W <= 0, both source forms or neither, n_cells out of the rule above, 7 * H * W > INT32_MAX (the largest distance),
 * and 2^31 tiles of 32 x 32 or more. */
int dm_geodesic_distance_i32(const uint8_t* traversable, const uint8_t* source_mask, const int64_t* source_cells,
                             int32_t n_cells, int32_t b, int32_t H, int32_t W, int32_t* dist, void* stream);

/* geodesic_path: per-environment paths from n start cells down a distance field (not in the reference).
 * traversable (b, H, W) u8 0 / 1 and dist (b, H, W) int32, normally dm_geodesic_distance_i32's output over that grid;
 * starts: device, (b, n, 2) int64 [x, z] = [column, row].  For start s of environment i, with D = dist[i] and
 * T = traversable[i]:
 *   1. if s lies outside the H x W map or D[s] < 0, the path is empty (length 0);
 *   2. otherwise p_0 = s.  While D[p_k] > 0 and k + 1 < max_cells, with d = D[p_k], the 8 neighbours
 *      q = p_k + (dx, dz) are tried in the fixed order (dx, dz) = (+1, 0), (0, +1), (-1, 0), (0, -1), (+1, +1),
 *      (-1, +1), (-1, -1), (+1, -1), and the first q with all of: q inside the map; D[q] >= 0; D[q] == d - c, c = 5
 *      for an orthogonal step and 7 for a diagonal one; the edge q -> p_k of dm_geodesic_distance_i32 (T[p_k], and for
 *      a diagonal step T[(q.x, p_k.z)] and T[(p_k.x, q.z)]) becomes p_k+1;
 *   3. the walk stops when D[p_k] == 0, when no neighbour qualifies, or when max_cells cells are written.
 * D strictly decreases along a walk, so it ends and visits distinct cells, at most min(max_cells, D[s] / 5 + 1) of
 * them, for any int32 dist.  When dist is the distance field of traversable, step 2 always finds a neighbour and the
 * path is a shortest path to a source: its step costs sum to D[s].
 * cells (b, n, max_cells, 2) int32 [x, z]: p_0 .. p_{len-1}, then -1, indexed in 64 bits; lengths (b, n) int32: len.
 * Every entry of both is written.  Exact integers.  One kernel on `stream`, no scratch, no atomics, no host
 * synchronisation; traversable, dist and starts are never written.  DM_EINVAL, before any CUDA call, for a null
 * pointer, b, H, W or n <= 0, H * W or b * n of 2^31 or more, and max_cells < 1 or > H * W. */
int dm_geodesic_path_i32(const uint8_t* traversable, const int32_t* dist, int32_t b, int32_t H, int32_t W,
                         const int64_t* starts, int32_t n, int32_t max_cells, int32_t* cells, int32_t* lengths,
                         void* stream);

/* connected_components: per-plane connected-component labels of masks (not in the reference).
 * mask (n_planes, H, W) u8, nonzero = foreground; each H x W plane is labelled on its own.  connectivity 4 (orthogonal
 * neighbours) or 8 (orthogonal and diagonal neighbours, no corner rule).
 * labels (n_planes, H, W) int32: 0 on background; the components of a plane are numbered 1..K in raster order of their
 * first cell (the smallest row * W + col), exactly as scipy.ndimage.label numbers them.  counts (n_planes) int32: K.
 * sizes (n_planes, H, W) int32, or NULL when not wanted: the cell count of each cell's component, 0 on background.
 * Deterministic whatever order the atomics run in.  Several kernels and a cub scan on `stream`, stream-ordered scratch
 * (cudaMallocAsync, 4 B a cell), no host synchronisation, no device-to-host copy; mask is never written.  DM_EINVAL,
 * before any CUDA call, for null mask, labels or counts, n_planes, H or W <= 0, connectivity not 4 or 8, and
 * n_planes * H * W > INT32_MAX. */
int dm_connected_components_i32(const uint8_t* mask, int32_t n_planes, int32_t H, int32_t W, int32_t connectivity,
                                int32_t* labels, int32_t* counts, int32_t* sizes, void* stream);

/* distance_transform: per-plane exact Euclidean distance transform of masks (not in the reference).
 * mask (n_planes, H, W) u8; each H x W plane is transformed on its own.
 * dist (n_planes, H, W) float32: 0 on zero cells; on nonzero cells the Euclidean distance in cells (centre to centre)
 * to the nearest zero cell of the plane, rounded as (float)sqrt((double)d2) from the exact integer squared distance d2,
 * which is exactly scipy.ndimage.distance_transform_edt(plane).astype(float32).
 * nearest (n_planes, H, W, 2) int32, or NULL when not wanted: [x, z] = [column, row] of a zero cell at exactly that
 * distance (the cell itself on zero cells); on ties one fixed such cell, the same on every call and whatever the other
 * planes hold.
 * A plane without a zero cell gets dist = +inf and nearest = -1 on every cell.  Two kernels on `stream`, stream-ordered
 * scratch (cudaMallocAsync, 2 B a cell), no atomics, no host synchronisation, no device-to-host copy; mask is never
 * written.  DM_EINVAL, before any CUDA call, for null mask or dist, n_planes, H or W <= 0, H or W > 32768 (d2 must fit
 * int32) and n_planes * H * W > INT32_MAX. */
int dm_distance_transform_f32(const uint8_t* mask, int32_t n_planes, int32_t H, int32_t W, float* dist,
                              int32_t* nearest, void* stream);

/* score_poses: per-environment match counts of a window against the planes of a global-frame map at candidate poses
 * (not in the reference; defined by its public functions).  For window cell (r, c) and candidate k of environment i:
 *   (lx, lz) = map_dequantize(c, r, window offsets, map_res, h, flip_h)
 *   (gx, gz) = local_to_global_space((lx, 0, lz), pose k)       (the DmStep of block i * n + k)
 *   (X, Z)   = map_quantize(gx, gz, source offsets, map_res, Hs, flip_h)
 * which is cell (r, c) of dm_crop_egocentric_f32 with that block, and
 *   scores[i, p, k] = #{(r, c) : window[i, p or 0, r, c] != 0, (X, Z) inside the source, planes[i, p, Z, X] != 0}.
 * planes (b, C, Hs, Ws) u8; window (b, window_planes, h, w) u8 with window_planes 1 (shared by the C planes) or C (one
 * per plane).  samples: device, b * n * DM_EGO_SAMPLE_WORDS floats from dm_pack_ego_samples, environment-major (block
 * i * n + k), each block with its own offsets.  scores (b, C, n) int32, every entry written.  Exact integer counts,
 * independent of evaluation order.  Two kernels on `stream` (counted as one launch), stream-ordered scratch
 * (cudaMallocAsync, 4 B per window cell), no atomics, no host synchronisation; planes, window and samples are never
 * written.  DM_EINVAL, before any CUDA call, for null pointers, b, C, Hs, Ws, h, w or n <= 0, window_planes not 1 or
 * C, map_res not > 0, b * n, h * w or Hs * Ws of 2^31 or more, and unaligned samples. */
int dm_score_poses_i32(const uint8_t* planes, int32_t b, int32_t C, int32_t Hs, int32_t Ws, float map_res,
                       int32_t flip_h, const uint8_t* window, int32_t window_planes, int32_t h, int32_t w,
                       const float* samples, int32_t n, int32_t* scores, void* stream);

/* visible_cells / count_visible: per-environment line of sight over masks from many origins (not in the reference).
 * blocking (b, H, W) u8, nonzero = blocks sight; origins: device, (b, n, 2) int64 [x, z] = [column, row].  For origin
 * o and target t = o + (dx, dz), with ax = |dx|, az = |dz|, m = max(ax, az) and sx, sz the signs of dx, dz, the line is
 * the cells p_i, i = 0..m, p_i = (ox + sx * i, oz + sz * floor((2 * i * az + m) / (2 * m))) when ax >= az and the same
 * with the axes swapped otherwise (p_0 = o, p_m = t).  t is visible from o when dx^2 + dz^2 <= radius^2, t is inside the
 * map, no p_i with 0 < i < m is blocking, and for no diagonal step p_i -> p_i+1 both side cells (x_i+1, z_i) and
 * (x_i, z_i+1) are blocking (no corner leak).  The origin and the target never block.  An origin outside the map sees
 * nothing.  Exactly one output:
 *   visible (b, n, 2r+1, 2r+1) u8: visible[i, k, r + dz, r + dx] = 1 iff o_ik + (dx, dz) is visible (targets NULL,
 *           C 0), indexed in 64 bits;
 *   counts  (b, C, n) int32: #{visible t : targets[i, c, t] != 0}, with targets (b, C, H, W) u8 and C >= 1.
 * Exact integers.  One kernel on `stream` (a memset of counts before it in count mode), no host synchronisation;
 * blocking, origins and targets are never written.  DM_EINVAL, before any CUDA call, for null blocking or origins, both
 * outputs or neither, targets without counts or the reverse, C not >= 1 with counts or not 0 without, b, H, W or
 * n <= 0, radius < 0 or > 512 (the staged window must fit in shared memory), and b * n, H * W or b * C * H * W of
 * 2^31 or more. */
int dm_line_of_sight_u8(const uint8_t* blocking, int32_t b, int32_t H, int32_t W, const int64_t* origins, int32_t n,
                        int32_t radius, uint8_t* visible, const uint8_t* targets, int32_t C, int32_t* counts,
                        void* stream);

/* Library/ABI introspection. */
int dm_abi_version(void);
/* sizeof() of a struct of this header as the library was compiled, for bindings to check their mirror against:
 * 0 DmStep, 1 DmProjSample, 2 DmProjCfg, 3 DmFlowSample, 4 DmFlowCfg, 5 DmFuseSource, 6 DmFuseTarget,
 * 7 DmBuilderCfg, 8 DmMapRef, 9 DmMergeShape, 10 DmPoseCfg, 11 DmValueMapRef; -1 for an unknown id. */
int32_t dm_sizeof_struct(int32_t id);
const char* dm_build_info(void);
/* Number of kernel launches issued by this library since load (bench "gpu_launches"). */
int64_t dm_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DUNGEON_MAPS_B200_H_ */
