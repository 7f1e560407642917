// MapBuilder.step with its host side in C: plot (orth_project with get_height_map, maps.py:2408-2469) + merge
// (fuse_topdown_maps, maps.py:2181-2287) for the case a mapping loop runs thousands of times — height maps of b
// environments, world map in the global frame.  The Python layer made ~1000 interpreter calls per step for a few
// hundred bytes of parameters (0.73 ms per step around 0.25 ms of merge kernels, profiles/r01n); here a step is two
// C calls: every parameter block (projection samples, the two fuse sources) is packed into ONE pinned staging slot,
// uploaded with ONE copy, and the kernels are launched back to back.  Nothing about the arithmetic changes: the
// rotation matrices are formed from sin / cos values the caller computes with the reference's own torch-CPU ops
// (utils.py:303-327; the last ulp matters), by the same float32 operations in the same order.
#include <cmath>
#include <cstring>
#include <new>

#include "dm_common.cuh"

namespace dm {
namespace {

constexpr int kParamSlots = 4;
constexpr int kStepWords = sizeof(DmStep) / 4;           // 16
constexpr int kSampleWords = sizeof(DmProjSample) / 4;   // 48
constexpr int kFuseWords = 2 * kStepWords + 2;           // per sample: two steps, width offset, height offset

}  // namespace
}  // namespace dm

using namespace dm;

struct DmBuilder {
  DmBuilderCfg cfg;      // value builders: cfg.proj.C channels, want_height set
  int C = 0;             // 0: height maps (dm_builder_create); >= 1: value maps (dm_builder_create_values)
  int labels = 0;        // value maps from class ids (dm_orth_project_labels_f32) instead of float planes
  int device = 0;
  DmPoseCfg pose;      // the constants of the yaw / pitch steps, fused as the projection's rotations are
  int fused_fuse = 0;  // DmStep.fused of the local map's local → global step in the merge
  int local_fast = 0;  // the pitch step has the structure DmProjCfg.fast_steps >= 1 promises
  char* h_params[kParamSlots] = {};
  char* d_params[kParamSlots] = {};
  cudaEvent_t ev[kParamSlots] = {};
  size_t param_bytes = 0;
  unsigned next = 0;
  int64_t* d_bbox = nullptr;
  int64_t* h_bbox = nullptr;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  // what dm_builder_plot leaves for dm_builder_merge
  DmFuseSource src[2];
  int n_src = 0;
  cudaEvent_t ev_bbox = nullptr;     // the bounding box has reached the host
  float* prefilled_top = nullptr;    // canvases dm_builder_plot_prefill filled while the host waited for the box
  float* prefilled_height = nullptr;  // (value maps: dm_builder_plot_values)
  uint8_t* prefilled_mask = nullptr;
  int64_t prefilled_cells = 0;
};

static void builder_free(DmBuilder* h) {
  if (!h) return;
  for (int i = 0; i < kParamSlots; ++i) {
    if (h->h_params[i]) cudaFreeHost(h->h_params[i]);
    if (h->d_params[i]) cudaFree(h->d_params[i]);
    if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  }
  if (h->ev_bbox) cudaEventDestroy(h->ev_bbox);
  if (h->d_bbox) cudaFree(h->d_bbox);
  if (h->h_bbox) cudaFreeHost(h->h_bbox);
  if (h->ws) cudaFree(h->ws);
  delete h;
}

static bool cfg_ok(const DmBuilderCfg* cfg, DmBuilder** out) {
  if (!cfg || !out || cfg->b <= 0) return false;
  if (cfg->proj.H <= 0 || cfg->proj.W <= 0 || cfg->proj.Mh <= 0 || cfg->proj.Mw <= 0) return false;
  return cfg->merge_reduction == 0 || cfg->merge_reduction == 1;
}

static int builder_create(const DmBuilderCfg* cfg, int C, int labels, int32_t device, DmBuilder** out);

extern "C" int dm_builder_create(const DmBuilderCfg* cfg, int32_t device, DmBuilder** out) {
  DM_TRACE();
  if (!cfg_ok(cfg, out) || cfg->proj.C != 0) return DM_EINVAL;
  return builder_create(cfg, 0, 0, device, out);
}

// MapBuilder.step(value_map=) / step(label_map=, num_classes=): the same step for C-channel value maps with their
// height planes (maps.py:335-349, 2258-2271).  Every argument is checked before the first CUDA call.
extern "C" int dm_builder_create_values(const DmBuilderCfg* cfg, int32_t labels, int32_t device, DmBuilder** out) {
  DM_TRACE();
  if (!cfg_ok(cfg, out) || cfg->proj.C < 1 || (labels && cfg->proj.C > 63)) return DM_EINVAL;
  if (cfg->proj.reduction != 0 && cfg->proj.reduction != 1) return DM_EINVAL;
  return builder_create(cfg, cfg->proj.C, labels ? 1 : 0, device, out);
}

static int builder_create(const DmBuilderCfg* cfg, int C, int labels, int32_t device, DmBuilder** out) {
  DmProjCfg pc = cfg->proj;
  pc.want_height = C > 0 ? 1 : 0;  // value maps: the local map's (b, 1, Mh, Mw) height plane too
  const size_t ws_bytes = labels ? dm_orth_project_labels_workspace_bytes(&pc, cfg->b)
                                 : dm_orth_project_workspace_bytes(&pc, cfg->b);
  if (ws_bytes == 0) return DM_EINVAL;
  DmBuilder* h = new (std::nothrow) DmBuilder();
  if (!h) return DM_EINVAL;
  h->cfg = *cfg;
  h->cfg.proj = pc;
  h->C = C;
  h->labels = labels;
  h->device = device;
  const long long n_proj = (long long)cfg->proj.H * cfg->proj.W;            // points one bmm rotates (utils.py:329)
  // C * h * w points of the local map (_fuse_source: local_to_global(pose, C * h * w)); a height map has one plane
  const long long n_fuse = (long long)(C > 0 ? C : 1) * cfg->proj.Mh * cfg->proj.Mw;
  memset(&h->pose, 0, sizeof(h->pose));
  memcpy(h->pose.pitch_R, cfg->pitch_R, sizeof(cfg->pitch_R));
  memcpy(h->pose.yaw_skew, cfg->yaw_skew, sizeof(cfg->yaw_skew));
  memcpy(h->pose.yaw_skew_sq, cfg->yaw_skew_sq, sizeof(cfg->yaw_skew_sq));
  h->pose.cam_height = cfg->cam_height;
  h->pose.fused = 9 * n_proj >= 400;
  h->fused_fuse = 9 * n_fuse >= 400;
  h->local_fast = local_step_is_fast(h->pose);
  h->param_bytes = ((size_t)cfg->b * (kSampleWords + 2 * kFuseWords) * 4 + 255) & ~(size_t)255;
  int rc = DM_OK;
#define DM_TRY(expr)                                                       \
  if (rc == DM_OK) {                                                       \
    const cudaError_t e_ = (expr);                                         \
    if (e_ != cudaSuccess) rc = static_cast<int>(e_);                      \
  }
  for (int i = 0; i < kParamSlots; ++i) {
    DM_TRY(cudaHostAlloc(reinterpret_cast<void**>(&h->h_params[i]), h->param_bytes, cudaHostAllocDefault));
    DM_TRY(cudaMalloc(reinterpret_cast<void**>(&h->d_params[i]), h->param_bytes));
    DM_TRY(cudaEventCreateWithFlags(&h->ev[i], cudaEventDisableTiming));
    if (!h->ev_bbox) DM_TRY(cudaEventCreateWithFlags(&h->ev_bbox, cudaEventDisableTiming));
  }
  DM_TRY(cudaMalloc(reinterpret_cast<void**>(&h->d_bbox), 5 * sizeof(int64_t)));
  DM_TRY(cudaHostAlloc(reinterpret_cast<void**>(&h->h_bbox), 5 * sizeof(int64_t), cudaHostAllocDefault));
  h->ws_bytes = ws_bytes;
  DM_TRY(cudaMalloc(&h->ws, h->ws_bytes));
  DM_TRY(cudaMemset(h->ws, 0, h->ws_bytes));
#undef DM_TRY
  if (rc != DM_OK) {
    builder_free(h);
    return rc;
  }
  *out = h;
  return DM_OK;
}

extern "C" void dm_builder_destroy(DmBuilder* h) { builder_free(h); }

// The packed parameter slot of a step, on the host and on the device:
//   [DmProjSample x b | local map's fuse params | world map's fuse params]
// and a source's fuse params are its steps (b, 2), width offsets (b) and height offsets (b).
struct FuseParams {
  float *steps, *woff, *hoff;
};

static FuseParams fuse_params(char* slot, int b, int source) {  // source 0: the local map, 1: the world map
  float* p = reinterpret_cast<float*>(slot) + (size_t)b * (kSampleWords + source * kFuseWords);
  return {p, p + (size_t)b * 2 * kStepWords, p + (size_t)b * (2 * kStepWords + 1)};
}

// Packs one step's parameter blocks into a pinned slot and queues their upload; returns the slot's device base.
// world: the world map whose offsets the merge uses, NULL without a world map
static int upload_params(DmBuilder* h, const float* pose, const float* sin_yaw, const float* cos_yaw,
                         const DmValueMapRef* world, cudaStream_t stream, char** d_base, int* fast_steps) {
  const DmBuilderCfg& c = h->cfg;
  const int b = c.b;
  const unsigned slot = h->next++ % kParamSlots;
  DM_CUDA_OK(cudaEventSynchronize(h->ev[slot]));  // the copy that last read this slot has run (it was queued long ago)
  float* samples = reinterpret_cast<float*>(h->h_params[slot]);
  const FuseParams lp = fuse_params(h->h_params[slot], b, 0), wp = fuse_params(h->h_params[slot], b, 1);
  int fast = h->local_fast ? (c.plot_to_global ? 2 : 1) : 0;
  for (int i = 0; i < b; ++i) {
    float Ry[9];
    yaw_matrix(h->pose, pose[3 * i + 2], sin_yaw[i], cos_yaw[i], Ry);  // utils.py:303-327 for the axis (0, 1, 0)
    const float ty[3] = {pose[3 * i + 0], 0.0f, pose[3 * i + 1]};  // maps.py:889-891
    const float tl[3] = {0.0f, c.cam_height, 0.0f};                // maps.py:795-797
    float* sp = samples + (size_t)i * kSampleWords;
    memset(sp, 0, sizeof(DmProjSample));
    put_step(sp, DM_STEP_ROT_THEN_ADD, c.pitch_R, tl, h->pose.fused);
    put_step(sp + kStepWords, c.plot_to_global ? DM_STEP_ROT_THEN_ADD : DM_STEP_NONE, Ry, ty, h->pose.fused);
    sp[32] = c.width_offset;
    sp[33] = c.height_offset;
    if (fast == 2 && !yaw_step_is_fast(Ry)) fast = 0;
    // the local map as a source of the merge (maps.py:2059-2060): local → global with its own pose, unless it was
    // plotted in the global frame; the target is global (maps.py:2116-2117: no second step)
    put_step(lp.steps + (size_t)i * 2 * kStepWords, c.plot_to_global ? DM_STEP_NONE : DM_STEP_ROT_THEN_ADD, Ry, ty,
             h->fused_fuse);
    put_step(lp.steps + (size_t)i * 2 * kStepWords + kStepWords, DM_STEP_NONE, nullptr, nullptr, 0);
    lp.woff[i] = c.width_offset;
    lp.hoff[i] = c.height_offset;
    put_step(wp.steps + (size_t)i * 2 * kStepWords, DM_STEP_NONE, nullptr, nullptr, 0);
    put_step(wp.steps + (size_t)i * 2 * kStepWords + kStepWords, DM_STEP_NONE, nullptr, nullptr, 0);
    wp.woff[i] = world ? world->width_offset : 0.0f;
    wp.hoff[i] = world ? world->height_offset : 0.0f;
  }
  DM_CUDA_OK(cudaMemcpyAsync(h->d_params[slot], h->h_params[slot], h->param_bytes, cudaMemcpyHostToDevice, stream));
  DM_CUDA_OK(cudaEventRecord(h->ev[slot], stream));
  *d_base = h->d_params[slot];
  *fast_steps = fast;
  return DM_OK;
}

// The fuse sources of a step: the old world map (NULL: none) first, then the local map.  A height builder's maps are
// their own height maps (world->height unused); a value builder's local map has one height plane for all C channels
// (the stride-0 expand of maps.py:349), its world map C planes of its own (maps.py:2258-2271).
static void make_sources(DmBuilder* h, char* d_base, float* local_topdown, uint8_t* local_mask, float* local_height,
                         const DmValueMapRef* world) {
  const DmBuilderCfg& c = h->cfg;
  const FuseParams lp = fuse_params(d_base, c.b, 0), wp = fuse_params(d_base, c.b, 1);
  h->n_src = 0;
  if (world) {  // fuse_topdown_maps(world, new): the world map first (maps.py:2471-2508)
    DmFuseSource& s = h->src[h->n_src++];
    const int64_t plane = (int64_t)world->h * world->w;
    if (h->C == 0) {
      s.height = world->topdown; s.values = nullptr;
      s.height_bstride = plane; s.height_cstride = plane;
    } else {
      s.height = world->height; s.values = world->topdown;
      s.height_bstride = plane * h->C; s.height_cstride = plane;
    }
    s.mask = world->mask;
    s.h = world->h; s.w = world->w; s.flip_h = c.proj.flip_h; s.map_res = c.proj.map_res;
    s.width_offset = wp.woff; s.height_offset = wp.hoff; s.steps = reinterpret_cast<const DmStep*>(wp.steps);
    s.plane_box = world->plane_box;
  }
  DmFuseSource& s = h->src[h->n_src++];
  s.mask = local_mask;
  s.height_bstride = (int64_t)c.proj.Mh * c.proj.Mw;
  if (h->C == 0) {
    s.height = local_topdown; s.values = nullptr; s.height_cstride = s.height_bstride;
  } else {
    s.height = local_height; s.values = local_topdown; s.height_cstride = 0;
  }
  s.h = c.proj.Mh; s.w = c.proj.Mw; s.flip_h = c.proj.flip_h; s.map_res = c.proj.map_res;
  s.width_offset = lp.woff; s.height_offset = lp.hoff; s.steps = reinterpret_cast<const DmStep*>(lp.steps);
  s.plane_box = nullptr;
}

// A height map as the shared code takes it: its topdown map is its height map (height NULL).
static DmValueMapRef value_ref(const DmMapRef& m) {
  DmValueMapRef v = {};
  v.topdown = m.topdown; v.height = nullptr; v.mask = m.mask; v.h = m.h; v.w = m.w;
  v.width_offset = m.width_offset; v.height_offset = m.height_offset;
  v.box = m.box; v.plane_box = m.plane_box;
  return v;
}

static DmFuseTarget fuse_target(const DmBuilder* h, const DmValueMapRef& m) {
  const DmBuilderCfg& c = h->cfg;
  DmFuseTarget t;
  t.Mh = m.h; t.Mw = m.w; t.flip_h = c.proj.flip_h; t.map_res = c.proj.map_res;
  t.width_offset = m.width_offset; t.height_offset = m.height_offset;
  t.fill_value = c.merge_fill_value; t.reduction = c.merge_reduction;
  return t;
}

// orth_project(get_height_map=True) of the step: local map and mask; value maps also their one height plane.
static int project_values(DmBuilder* h, const float* depth, const float* values, const uint8_t* labels, char* d_base,
                          int fast, float* topdown, uint8_t* mask, float* height, cudaStream_t stream) {
  DmProjCfg pc = h->cfg.proj;
  pc.fast_steps = fast;
  const DmProjSample* samples = reinterpret_cast<const DmProjSample*>(d_base);
  if (h->labels)
    return dm_orth_project_labels_f32(depth, labels, nullptr, samples, &pc, h->cfg.b, topdown, mask, height, h->ws,
                                      h->ws_bytes, stream);
  return dm_orth_project_f32(depth, values, nullptr, samples, &pc, h->cfg.b, topdown, mask, height, h->ws, h->ws_bytes,
                             stream);
}

// The first half of a step for both kinds of handle (height maps: values, labels, local_height and every height NULL):
// projection, bounding box of world ∪ local, its copy to the host, and the fill of the canvases the caller guessed.
static int builder_plot(DmBuilder* h, const float* depth, const float* values, const uint8_t* labels, const float* pose,
                        const float* sin_yaw, const float* cos_yaw, float* local_topdown, uint8_t* local_mask,
                        float* local_height, const DmValueMapRef* world, DmMergeShape* shape, float* prefill_topdown,
                        float* prefill_height, uint8_t* prefill_mask, int64_t prefill_cells, cudaStream_t stream) {
  char* d_base = nullptr;
  int fast = 0;
  int rc = upload_params(h, pose, sin_yaw, cos_yaw, world, stream, &d_base, &fast);
  if (rc != DM_OK) return rc;
  make_sources(h, d_base, local_topdown, local_mask, local_height, world);
  // pass 1 (maps.py:2146-2179): a world map that carries the box its own scatter pass tracked only seeds the reduction
  const bool seeded = world && world->box;
  bool fused = false;
  if (h->C == 0) {
    // the projection's resolve pass and pass 1 over the local map it writes are ONE kernel (dm_fuse.cu:
    // hmap_resolve_bbox_kernel) whenever the depth-only projection can hand over its key planes
    DmProjCfg pc = h->cfg.proj;
    pc.fast_steps = fast;
    uint32_t* planes = nullptr;
    unsigned long long slot_words = 0;
    rc = hmap_project_keys(depth, nullptr, reinterpret_cast<const DmProjSample*>(d_base), &pc, h->cfg.b, h->ws,
                           h->ws_bytes, stream, &planes, &slot_words);
    if (rc != DM_OK && rc != DM_EINVAL) return rc;
    fused = rc == DM_OK;
    if (fused) {
      rc = hmap_resolve_with_bbox(planes, slot_words, &pc, h->cfg.b, local_topdown, local_mask, &h->src[h->n_src - 1],
                                  h->cfg.proj.map_res, seeded ? world->box : nullptr, h->d_bbox, stream);
      if (rc != DM_OK) return rc;
      if (world && !seeded) {  // an untracked world map is scanned as before
        rc = fuse_bbox_accumulate(h->src, 1, h->cfg.b, 1, h->cfg.proj.map_res, h->d_bbox, stream);
        if (rc != DM_OK) return rc;
      }
    }
  }
  if (!fused) {  // value maps, and height maps of more than 64 frames or with the height-map path switched off
    rc = project_values(h, depth, values, labels, d_base, fast, local_topdown, local_mask, local_height, stream);
    if (rc != DM_OK) return rc;
    const DmFuseSource* scan = seeded ? &h->src[h->n_src - 1] : h->src;
    rc = dm_fuse_bbox_seeded_i64(scan, seeded ? 1 : h->n_src, h->cfg.b, h->C > 0 ? h->C : 1, h->cfg.proj.map_res,
                                 seeded ? world->box : nullptr, h->d_bbox, stream);
    if (rc != DM_OK) return rc;
  }
  DM_CUDA_OK(cudaMemcpyAsync(h->h_bbox, h->d_bbox, 5 * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  DM_CUDA_OK(cudaEventRecord(h->ev_bbox, stream));
  h->prefilled_top = nullptr; h->prefilled_height = nullptr; h->prefilled_mask = nullptr; h->prefilled_cells = 0;
  prefill_cells &= ~(int64_t)15;
  if (prefill_topdown && prefill_mask && (h->C == 0 || prefill_height) && prefill_cells > 0) {
    rc = dm_fuse_canvas_init_f32(prefill_topdown, prefill_mask, prefill_height, prefill_cells, h->cfg.merge_fill_value,
                                 stream);
    if (rc != DM_OK) return rc;
    h->prefilled_top = prefill_topdown; h->prefilled_height = prefill_height; h->prefilled_mask = prefill_mask;
    h->prefilled_cells = prefill_cells;
  }
  return shape ? dm_builder_plot_wait(h, shape) : DM_OK;  // shape == NULL: the caller waits later (dm_builder_plot_wait)
}

// The second half: fills `out` and scatters the sources builder_plot left into it.
static int builder_merge(DmBuilder* h, const DmValueMapRef& out, void* stream) {
  const DmBuilderCfg& c = h->cfg;
  const int planes = h->C > 0 ? h->C : 1;
  const DmFuseTarget tgt = fuse_target(h, out);
  // the prefill covers the first prefilled_cells cells (a multiple of 16: the tail below starts 16-byte aligned) of the
  // canvases the caller guessed; a map that outgrew the guess gets its tail filled here
  const int64_t n_cells = (int64_t)c.b * planes * out.h * out.w;  // 64-bit: b * C * h * w passes 2^31 at scale
  const bool prefilled = out.topdown == h->prefilled_top && out.height == h->prefilled_height &&
                         out.mask == h->prefilled_mask && h->prefilled_cells > 0;
  if (prefilled && n_cells > h->prefilled_cells) {
    const int64_t p = h->prefilled_cells;
    const int rf = dm_fuse_canvas_init_f32(out.topdown + p, out.mask + p, out.height ? out.height + p : nullptr,
                                           n_cells - p, c.merge_fill_value, stream);
    if (rf != DM_OK) return rf;
  }
  const int rc = fuse_scatter_track(h->src, h->n_src, c.b, planes, &tgt, out.topdown, out.mask, out.height, out.box,
                                    out.plane_box, prefilled ? 1 : 0, stream);
  h->prefilled_top = nullptr; h->prefilled_height = nullptr; h->prefilled_mask = nullptr; h->prefilled_cells = 0;
  h->n_src = 0;
  return rc;
}

// The fixed-canvas step: plot, then merge in place.  For a height handle project_values is the depth-only projection
// (want_height 0, values and labels NULL).
static int builder_step_fixed(DmBuilder* h, const float* depth, const float* values, const uint8_t* labels,
                              const float* pose, const float* sin_yaw, const float* cos_yaw, float* local_topdown,
                              uint8_t* local_mask, float* local_height, const DmValueMapRef& canvas,
                              cudaStream_t stream) {
  char* d_base = nullptr;
  int fast = 0;
  int rc = upload_params(h, pose, sin_yaw, cos_yaw, nullptr, stream, &d_base, &fast);
  if (rc != DM_OK) return rc;
  rc = project_values(h, depth, values, labels, d_base, fast, local_topdown, local_mask, local_height, stream);
  if (rc != DM_OK) return rc;
  make_sources(h, d_base, local_topdown, local_mask, local_height, nullptr);
  const DmFuseTarget tgt = fuse_target(h, canvas);
  rc = dm_fuse_inplace_f32(h->src, 1, h->cfg.b, h->C > 0 ? h->C : 1, &tgt, canvas.topdown, canvas.mask, canvas.height,
                           stream);
  h->n_src = 0;
  return rc;
}

// ---- height maps (dm_builder_create) ------------------------------------------------------------------------------

static bool height_map_ok(const DmMapRef* m) { return m->topdown && m->mask && m->h > 0 && m->w > 0; }

extern "C" int dm_builder_plot(DmBuilder* h, const float* depth, const float* pose, const float* sin_yaw,
                               const float* cos_yaw, float* local_topdown, uint8_t* local_mask, const DmMapRef* world,
                               DmMergeShape* shape, void* stream_) {
  DM_TRACE();
  return dm_builder_plot_prefill(h, depth, pose, sin_yaw, cos_yaw, local_topdown, local_mask, world, shape, nullptr,
                                 nullptr, 0, stream_);
}

// dm_builder_plot + speculation: the GPU is idle from the moment the bounding box is on its way to the host until the
// merge kernels are queued (copy latency, the host computing the canvas shape, five launches) — ~55 us of a 316 us step.
// The canvas of the merge is as a rule in the size class of the old world map, so the caller hands canvases of that
// class in BEFORE the box is known: the fill (the largest merge kernel, 115 us) is queued right behind the box's copy
// and runs while the host waits for the box and prepares the scatter launches.  dm_builder_merge skips its fill when
// `out` is what was prefilled (and large enough); anything else is filled as before.
extern "C" int dm_builder_plot_prefill(DmBuilder* h, const float* depth, const float* pose, const float* sin_yaw,
                                       const float* cos_yaw, float* local_topdown, uint8_t* local_mask,
                                       const DmMapRef* world, DmMergeShape* shape, float* prefill_topdown,
                                       uint8_t* prefill_mask, int64_t prefill_cells, void* stream_) {
  DM_TRACE();
  if (!h || h->C != 0 || !depth || !pose || !sin_yaw || !cos_yaw || !local_topdown || !local_mask) return DM_EINVAL;
  if (world && !height_map_ok(world)) return DM_EINVAL;
  const DmValueMapRef wv = world ? value_ref(*world) : DmValueMapRef{};
  return builder_plot(h, depth, nullptr, nullptr, pose, sin_yaw, cos_yaw, local_topdown, local_mask, nullptr,
                      world ? &wv : nullptr, shape, prefill_topdown, nullptr, prefill_mask, prefill_cells,
                      static_cast<cudaStream_t>(stream_));
}

extern "C" int dm_builder_plot_wait(DmBuilder* h, DmMergeShape* shape) {
  DM_TRACE();
  if (!h || !shape) return DM_EINVAL;
  DM_CUDA_OK(cudaEventSynchronize(h->ev_bbox));  // the reference's .item() sync (maps.py:2172-2173)
  const int64_t min_x = h->h_bbox[0], max_x = h->h_bbox[1], min_z = h->h_bbox[2], max_z = h->h_bbox[3];
  shape->n_valid = h->h_bbox[4];
  if (shape->n_valid == 0) return DM_OK;  // maps.py:2217-2225: the caller keeps the last map
  // maps.py:2171-2178: sizes as Python ints, offsets as float32 tensors
  const int64_t map_width = (max_x - min_x) + 2, map_height = (max_z - min_z) + 2;
  if (map_width <= 0 || map_height <= 0 || map_width >= (1ll << 31) || map_height >= (1ll << 31)) return DM_EINVAL;
  shape->map_width = (int32_t)map_width;
  shape->map_height = (int32_t)map_height;
  shape->width_offset = (float)((double)map_width / 2.0) - (float)(max_x + min_x) / 2.0f;
  shape->height_offset = (float)((double)map_height / 2.0) - (float)(max_z + min_z) / 2.0f;
  return DM_OK;
}

extern "C" int dm_builder_merge(DmBuilder* h, const DmMapRef* out, void* stream_) {
  DM_TRACE();
  if (!h || h->C != 0 || !out || !height_map_ok(out) || h->n_src <= 0) return DM_EINVAL;
  return builder_merge(h, value_ref(*out), stream_);
}

extern "C" int dm_builder_step_fixed(DmBuilder* h, const float* depth, const float* pose, const float* sin_yaw,
                                     const float* cos_yaw, float* local_topdown, uint8_t* local_mask,
                                     const DmMapRef* canvas, void* stream_) {
  DM_TRACE();
  if (!h || h->C != 0 || !depth || !pose || !sin_yaw || !cos_yaw || !local_topdown || !local_mask) return DM_EINVAL;
  if (!canvas || !height_map_ok(canvas)) return DM_EINVAL;
  return builder_step_fixed(h, depth, nullptr, nullptr, pose, sin_yaw, cos_yaw, local_topdown, local_mask, nullptr,
                            value_ref(*canvas), static_cast<cudaStream_t>(stream_));
}

// ---- value maps (dm_builder_create_values) ----------------------------------------------------------------------

static bool value_inputs_ok(const DmBuilder* h, const float* depth, const float* values, const uint8_t* labels,
                            const float* pose, const float* sin_yaw, const float* cos_yaw, const float* local_topdown,
                            const uint8_t* local_mask, const float* local_height) {
  if (!h || h->C == 0 || !depth || !pose || !sin_yaw || !cos_yaw || !local_topdown || !local_mask || !local_height)
    return false;
  return h->labels ? (labels && !values) : (values && !labels);
}

static bool value_map_ok(const DmValueMapRef* m) {
  return m->topdown && m->height && m->mask && m->h > 0 && m->w > 0;
}

extern "C" int dm_builder_plot_values(DmBuilder* h, const float* depth, const float* values, const uint8_t* labels,
                                      const float* pose, const float* sin_yaw, const float* cos_yaw,
                                      float* local_topdown, uint8_t* local_mask, float* local_height,
                                      const DmValueMapRef* world, DmMergeShape* shape, float* prefill_topdown,
                                      float* prefill_height, uint8_t* prefill_mask, int64_t prefill_cells,
                                      void* stream_) {
  DM_TRACE();
  if (!value_inputs_ok(h, depth, values, labels, pose, sin_yaw, cos_yaw, local_topdown, local_mask, local_height))
    return DM_EINVAL;
  if (world && !value_map_ok(world)) return DM_EINVAL;
  return builder_plot(h, depth, values, labels, pose, sin_yaw, cos_yaw, local_topdown, local_mask, local_height, world,
                      shape, prefill_topdown, prefill_height, prefill_mask, prefill_cells,
                      static_cast<cudaStream_t>(stream_));
}

extern "C" int dm_builder_merge_values(DmBuilder* h, const DmValueMapRef* out, void* stream_) {
  DM_TRACE();
  if (!h || h->C == 0 || !out || !value_map_ok(out) || h->n_src <= 0) return DM_EINVAL;
  return builder_merge(h, *out, stream_);
}

extern "C" int dm_builder_step_fixed_values(DmBuilder* h, const float* depth, const float* values,
                                            const uint8_t* labels, const float* pose, const float* sin_yaw,
                                            const float* cos_yaw, float* local_topdown, uint8_t* local_mask,
                                            float* local_height, const DmValueMapRef* canvas, void* stream_) {
  DM_TRACE();
  if (!value_inputs_ok(h, depth, values, labels, pose, sin_yaw, cos_yaw, local_topdown, local_mask, local_height))
    return DM_EINVAL;
  if (!canvas || !value_map_ok(canvas)) return DM_EINVAL;
  return builder_step_fixed(h, depth, values, labels, pose, sin_yaw, cos_yaw, local_topdown, local_mask, local_height,
                            *canvas, static_cast<cudaStream_t>(stream_));
}
