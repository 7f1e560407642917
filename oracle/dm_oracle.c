/*
 * ORACLE — TEST INFRASTRUCTURE ONLY.  Not part of the product.
 *
 * Scalar CPU restatement of the reference's depth → top-down hot path
 * (Ending2015a/dungeon_maps v0.0.3a1).  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load this.
 *
 * Parity is PINNED: tests/test_oracle_golden.py checks every function here
 * bit-for-bit against tests/golden/ (npz files), which oracle/make_golden.py produced
 * by running the unmodified reference (imported from /root/reference through
 * the torch_scatter stand-in in oracle/ref_shim.py) on CPU.
 *
 * All arithmetic is float32 with one rounding per reference torch op.
 * Build: gcc -O2 -ffp-contract=off -mfma -fopenmp -shared -fPIC (see oracle/build.py);
 * -ffp-contract=off forbids the compiler from fusing a*b+c on its own, fmaf()
 * is used exactly where the reference's sgemm (torch.einsum → bmm → MKL) fused.
 *
 * Struct layouts come from include/dungeon_maps_b200.h (layout only; no code is shared
 * with the CUDA library).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../include/dungeon_maps_b200.h"

#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct { float x, y, z; } vec3;

/* utils.py:329  torch.einsum('bji,b...j->b...i', R, points) → at::bmm on CPU
 * (ATen LinearAlgebra.cpp bmm_out_or_baddbmm_): for contraction*rows*cols = 9*n >= 400 it is
 * MKL sgemm, which accumulates j = 0,1,2 with FMA: fma(R2i,p2, fma(R1i,p1, rn(R0i*p0)));
 * below that it is ATen's naive triple loop compiled without FMA: ((R0i*p0 + R1i*p1) + R2i*p2).
 * Both were established by probing the reference (oracle/make_golden.py N = 1..1000). */
static inline vec3 rot(const float* R, vec3 p, int fused) {
  vec3 o;
  if (fused) {
    o.x = fmaf(R[6], p.z, fmaf(R[3], p.y, R[0] * p.x));
    o.y = fmaf(R[7], p.z, fmaf(R[4], p.y, R[1] * p.x));
    o.z = fmaf(R[8], p.z, fmaf(R[5], p.y, R[2] * p.x));
  } else {
    o.x = (R[0] * p.x + R[3] * p.y) + R[6] * p.z;
    o.y = (R[1] * p.x + R[4] * p.y) + R[7] * p.z;
    o.z = (R[2] * p.x + R[5] * p.y) + R[8] * p.z;
  }
  return o;
}

/* utils.py:229-259 translate: points + offsets (all three components are added,
 * zeros included). */
static inline vec3 add3(vec3 p, const float* t) {
  vec3 o = {p.x + t[0], p.y + t[1], p.z + t[2]};
  return o;
}

/* maps.py:753-942: the four space transforms are a rotate and a translate in
 * one order or the other. */
static inline vec3 apply_step(const DmStep* s, vec3 p) {
  if (s->kind == DM_STEP_ROT_THEN_ADD) return add3(rot(s->R, p, s->fused), s->t);
  if (s->kind == DM_STEP_ADD_THEN_ROT) return rot(s->R, add3(p, s->t), s->fused);
  if (s->kind == DM_STEP_ADD) return add3(p, s->t);
  if (s->kind == DM_STEP_ROT) return rot(s->R, p, s->fused);
  return p;
}

/* Tensor.to(int64) of a float on x86 (cvttss2si): NaN / out of range → INT64_MIN. */
static inline int64_t f2i64(float v) {
  if (!(v >= -9223372036854775808.0f && v < 9223372036854775808.0f)) return INT64_MIN;
  return (int64_t)v;
}

/* maps.py:1004-1013 map_quantize for one point. */
static inline void quantize1(float x, float z, float woff, float hoff, float res, int32_t Mh,
                             int32_t flip_h, int64_t* xi, int64_t* zi) {
  float xb = x / res + woff;
  float zb = z / res + hoff;
  if (flip_h) zb = (float)(Mh - 1) - zb;
  *xi = f2i64(floorf(xb + 0.5f));
  *zi = f2i64(floorf(zb + 0.5f));
}

/* maps.py:667-679 image_to_camera_space for pixel (row r, col c) of an H-row frame. */
static inline vec3 unproject(int r, int c, float z, int H, float fx, float fy, float cx, float cy,
                             int flip_h) {
  float yy = flip_h ? (float)(H - 1) - (float)r : (float)r;
  vec3 p;
  p.x = ((float)c - cx) / fx * z;
  p.y = (yy - cy) / fy * z;
  p.z = z;
  return p;
}

static inline int better(float v, float cur, int reduction) {
  /* torch_scatter CPU: `if (src > out) out = src` (max) / `<` (min); NaN never wins. */
  return reduction == 0 ? (v > cur) : (v < cur);
}

/* utils.py:489-491: mask = nan_to_num(|new - old|) != 0 with old == fill everywhere. */
static inline uint8_t changed(float now, float fill) {
  float d = fabsf(now - fill);
  if (isnan(d)) d = 0.0f;
  return d != 0.0f;
}

/* orth_project, maps.py:127-351.  Shapes as dm_orth_project_f32 (host pointers). */
int dmo_orth_project(const float* depth, const float* values, const uint8_t* valid,
                     const DmProjSample* samples, const DmProjCfg* cfg, int32_t b, float* topdown,
                     uint8_t* mask, float* height, int32_t threads) {
  const int H = cfg->H, W = cfg->W, C = cfg->C, Mh = cfg->Mh, Mw = cfg->Mw;
  const int Cout = C > 0 ? C : 1;
  const int64_t N = (int64_t)H * W, M = (int64_t)Mh * Mw;
  const float ninf = -INFINITY;
  const int want_h = (C > 0 && cfg->want_height && height != NULL);
#ifdef _OPENMP
  if (threads > 0) omp_set_num_threads(threads);
#endif
#pragma omp parallel for schedule(dynamic, 1)
  for (int32_t s = 0; s < b; ++s) {
    const DmProjSample* sp = &samples[s];
    const float* d = depth + (int64_t)s * N;
    const uint8_t* vm = valid ? valid + (int64_t)s * N : NULL;
    float* top = topdown + (int64_t)s * Cout * M;
    float* hgt = want_h ? height + (int64_t)s * M : NULL;
    /* utils.py:472-474: canvas.fill_(fill_value) (zeros when None) */
    for (int64_t i = 0; i < Cout * M; ++i) top[i] = cfg->fill_value;
    if (hgt) for (int64_t i = 0; i < M; ++i) hgt[i] = ninf; /* maps.py:345 */
    for (int r = 0; r < H; ++r) {
      for (int c = 0; c < W; ++c) {
        const int64_t px = (int64_t)r * W + c;
        const float z = d[px];
        /* maps.py:537-544 */
        int ok = 1;
        if (cfg->has_trunc_depth_max) ok &= (z <= cfg->trunc_depth_max);
        if (cfg->has_trunc_depth_min) ok &= (z >= cfg->trunc_depth_min);
        if (vm) ok &= (vm[px] != 0);
        /* maps.py:48-70, 273-277 */
        if (cfg->clip_border > 0) {
          const int k = cfg->clip_border;
          ok &= (r >= k) & (r < H - k) & (c >= k) & (c < W - k);
        }
        vec3 p = unproject(r, c, z, H, cfg->fx, cfg->fy, cfg->cx, cfg->cy, cfg->flip_h);
        p = apply_step(&sp->to_local, p); /* maps.py:279-284 */
        if (cfg->has_trunc_height_max) ok &= (p.y <= cfg->trunc_height_max); /* maps.py:286-288 */
        p = apply_step(&sp->to_global, p); /* maps.py:290-295 */
        int64_t xi, zi;
        quantize1(p.x, p.z, sp->width_offset, sp->height_offset, cfg->map_res, Mh, cfg->flip_h,
                  &xi, &zi); /* maps.py:301-310 */
        ok &= (xi >= 0) & (xi < Mw) & (zi >= 0) & (zi < Mh); /* maps.py:1155-1158 */
        if (!ok) continue;
        const int64_t cell = zi * Mw + xi; /* utils.py:332-370 */
        if (C == 0) {
          if (better(p.y, top[cell], cfg->reduction)) top[cell] = p.y;
        } else {
          const float* v = values + (int64_t)s * C * N + px;
          for (int ch = 0; ch < C; ++ch) {
            const float val = v[(int64_t)ch * N];
            float* t = &top[(int64_t)ch * M + cell];
            if (better(val, *t, cfg->reduction)) *t = val;
          }
          if (hgt && p.y > hgt[cell]) hgt[cell] = p.y; /* maps.py:340-348, always max */
        }
      }
    }
    uint8_t* mk = mask + (int64_t)s * Cout * M;
    for (int64_t i = 0; i < Cout * M; ++i) mk[i] = changed(top[i], cfg->fill_value);
  }
  return 0;
}

/* camera_affine_grid, maps.py:353-460 (+ demo compute_ego_flow when cfg->emit_flow). */
int dmo_affine_grid(const float* depth, const DmFlowSample* samples, const DmFlowCfg* cfg,
                    int32_t b, float* grid, int32_t threads) {
  const int H = cfg->H, W = cfg->W, CH = cfg->channels;
  const int64_t N = (int64_t)H * W;
#ifdef _OPENMP
  if (threads > 0) omp_set_num_threads(threads);
#endif
#pragma omp parallel for schedule(dynamic, 1) collapse(2)
  for (int32_t s = 0; s < b; ++s) {
    for (int ch = 0; ch < CH; ++ch) {
      const DmFlowSample* sp = &samples[s];
      const float* d = depth + ((int64_t)s * CH + ch) * N;
      float* g = grid + ((int64_t)s * CH + ch) * N * 2;
      for (int r = 0; r < H; ++r) {
        for (int c = 0; c < W; ++c) {
          const int64_t px = (int64_t)r * W + c;
          vec3 p = unproject(r, c, d[px], H, cfg->fx, cfg->fy, cfg->cx, cfg->cy, cfg->flip_h);
          p = apply_step(&sp->to_local, p);
          p = apply_step(&sp->transition, p);
          p = apply_step(&sp->to_camera, p);
          /* maps.py:743-747 camera_to_image_space */
          const float ze = p.z + 1e-7f;
          float gx = p.x / ze * cfg->fx + cfg->cx;
          float gy = p.y / ze * cfg->fy + cfg->cy;
          if (cfg->flip_h) gy = (float)(H - 1) - gy;
          if (cfg->emit_flow) { /* demos/ego_flow/run.py:86-89 */
            gx = (float)c - gx;
            gy = -((float)r - gy);
          }
          g[px * 2 + 0] = gx;
          g[px * 2 + 1] = gy;
        }
      }
    }
  }
  return 0;
}

/* points (b, n, 3): apply steps[b][n_steps] in order. */
int dmo_transform_points(const float* points, const DmStep* steps, int32_t n_steps, int32_t b,
                         int64_t n, float* out) {
  for (int32_t s = 0; s < b; ++s)
    for (int64_t i = 0; i < n; ++i) {
      const float* q = points + ((int64_t)s * n + i) * 3;
      vec3 p = {q[0], q[1], q[2]};
      for (int k = 0; k < n_steps; ++k) p = apply_step(&steps[s * n_steps + k], p);
      float* o = out + ((int64_t)s * n + i) * 3;
      o[0] = p.x; o[1] = p.y; o[2] = p.z;
    }
  return 0;
}

/* maps.py:616-682 / 684-751 on (n,3) points. */
int dmo_image_camera(const float* points, int64_t n, float fx, float fy, float cx, float cy,
                     int32_t flip_h, int32_t height, int32_t to_image, float* out) {
  for (int64_t i = 0; i < n; ++i) {
    float x = points[i * 3], y = points[i * 3 + 1], z = points[i * 3 + 2];
    if (!to_image) {
      if (flip_h) y = (float)(height - 1) - y;
      x = (x - cx) / fx * z;
      y = (y - cy) / fy * z;
    } else {
      const float ze = z + 1e-7f;
      x = x / ze * fx + cx;
      y = y / ze * fy + cy;
      if (flip_h) y = (float)(height - 1) - y;
    }
    out[i * 3] = x; out[i * 3 + 1] = y; out[i * 3 + 2] = z;
  }
  return 0;
}

/* maps.py:462-545 */
int dmo_depth_to_points(const float* depth, const uint8_t* valid_in, int64_t frames, int32_t H,
                        int32_t W, float fx, float fy, float cx, float cy, int32_t flip_h,
                        int32_t has_tmin, float tmin, int32_t has_tmax, float tmax, float* points,
                        uint8_t* valid_out) {
  const int64_t N = (int64_t)H * W;
  for (int64_t f = 0; f < frames; ++f)
    for (int r = 0; r < H; ++r)
      for (int c = 0; c < W; ++c) {
        const int64_t i = f * N + (int64_t)r * W + c;
        const float z = depth[i];
        vec3 p = unproject(r, c, z, H, fx, fy, cx, cy, flip_h);
        points[i * 3] = p.x; points[i * 3 + 1] = p.y; points[i * 3 + 2] = p.z;
        int ok = 1;
        if (has_tmax) ok &= (z <= tmax);
        if (has_tmin) ok &= (z >= tmin);
        if (valid_in) ok &= (valid_in[i] != 0);
        valid_out[i] = (uint8_t)ok;
      }
  return 0;
}

/* maps.py:944-1019 */
int dmo_map_quantize(const float* x, const float* z, const float* woff, const float* hoff,
                     int32_t b, int64_t n, float res, int32_t Mh, int32_t flip_h, int64_t* xb,
                     int64_t* zb) {
  for (int32_t s = 0; s < b; ++s)
    for (int64_t i = 0; i < n; ++i)
      quantize1(x[s * n + i], z[s * n + i], woff[s], hoff[s], res, Mh, flip_h, &xb[s * n + i],
                &zb[s * n + i]);
  return 0;
}

/* maps.py:1021-1087 */
int dmo_map_dequantize(const float* xb, const float* zb, const float* woff, const float* hoff,
                       int32_t b, int64_t n, float res, int32_t Mh, int32_t flip_h, float* x,
                       float* z) {
  for (int32_t s = 0; s < b; ++s)
    for (int64_t i = 0; i < n; ++i) {
      float zz = zb[s * n + i];
      if (flip_h) zz = (float)(Mh - 1) - zz;
      z[s * n + i] = (zz - hoff[s]) * res;
      x[s * n + i] = (xb[s * n + i] - woff[s]) * res;
    }
  return 0;
}

/* utils.py:389-492 for a 2-D canvas; coords (B, N, 2) = [row, col]. */
int dmo_scatter(const float* values, const int64_t* coords, const uint8_t* valid, int64_t B,
                int64_t N, int32_t Mh, int32_t Mw, int32_t has_fill, float fill, int32_t reduction,
                float* canvas, uint8_t* mask) {
  /* reduction (utils.py:44-76): 0 max, 1 min, 2 sum, 3 mean, 4 prod; hits are applied in index order like
   * torch_scatter's CPU loops.  mean (torch_scatter.scatter_mean with out=): the starting canvas takes part in
   * the sum, not in the count; count is clamped to >= 1.  torch_scatter counts with a scatter_add_ of float32 ones:
   * that count stops at 2^24 (2^24 + 1 rounds back to 2^24), so the divisor is min(count, 2^24). */
  const int64_t M = (int64_t)Mh * Mw;
  float* before = (float*)malloc(sizeof(float) * (size_t)M);
  int32_t* count = (int32_t*)malloc(sizeof(int32_t) * (size_t)M);
  if (!before || !count) { free(before); free(count); return -1; }
  for (int64_t s = 0; s < B; ++s) {
    float* cv = canvas + s * M;
    if (has_fill) for (int64_t i = 0; i < M; ++i) cv[i] = fill;
    memcpy(before, cv, sizeof(float) * (size_t)M);
    memset(count, 0, sizeof(int32_t) * (size_t)M);
    for (int64_t i = 0; i < N; ++i) {
      if (valid && !valid[s * N + i]) continue;
      const int64_t r = coords[(s * N + i) * 2], c = coords[(s * N + i) * 2 + 1];
      if (r < 0 || r >= Mh || c < 0 || c >= Mw) continue;
      float* t = &cv[r * Mw + c];
      const float v = values[s * N + i];
      if (reduction == 2 || reduction == 3) { *t = *t + v; count[r * Mw + c] += 1; }
      else if (reduction == 4) *t = *t * v;
      else if (better(v, *t, reduction)) *t = v;
    }
    if (reduction == 3)
      for (int64_t i = 0; i < M; ++i)
        cv[i] = cv[i] / (count[i] < 1 ? 1.0f : count[i] < (1 << 24) ? (float)count[i] : 16777216.0f);
    for (int64_t i = 0; i < M; ++i) {
      float d = fabsf(cv[i] - before[i]);
      if (isnan(d)) d = 0.0f;
      mask[s * M + i] = d != 0.0f;
    }
  }
  free(before);
  free(count);
  return 0;
}

/* fuse_topdown_maps, maps.py:2039-2127: every cell of one source map as a point in the
 * target frame.  height (b, C, h, w) with explicit batch/channel strides.
 * Outputs px, pz (b, C, h*w) f32. */
int dmo_fuse_points(const float* height, int64_t bstride, int64_t cstride, int32_t b, int32_t C,
                    int32_t h, int32_t w, int32_t flip_h, float res, const float* woff,
                    const float* hoff, const DmStep* steps /* (b,2) */, float* px, float* py,
                    float* pz) {
  const int64_t n = (int64_t)h * w;
  for (int32_t s = 0; s < b; ++s)
    for (int32_t ch = 0; ch < C; ++ch)
      for (int r = 0; r < h; ++r)
        for (int c = 0; c < w; ++c) {
          /* maps.py:1081-1086 map_dequantize */
          float zb = (float)r;
          if (flip_h) zb = (float)(h - 1) - zb;
          vec3 p;
          p.z = (zb - hoff[s]) * res;
          p.x = ((float)c - woff[s]) * res;
          p.y = height[s * bstride + ch * cstride + (int64_t)r * w + c];
          p = apply_step(&steps[s * 2 + 0], p);
          p = apply_step(&steps[s * 2 + 1], p);
          const int64_t o = ((int64_t)s * C + ch) * n + (int64_t)r * w + c;
          px[o] = p.x; py[o] = p.y; pz[o] = p.z;
        }
  return 0;
}

/* crop_topdown_map, maps.py:1959-2037: generate_crop_grid (utils.py:571-611) followed by
 * image_sample (utils.py:613-652) = F.pad(1, fill) + F.grid_sample(nearest,
 * align_corners=True, padding_mode = border if fill given else zeros), as ATen's
 * vectorised CPU kernel evaluates it. */
int dmo_crop_nearest(const float* image, const float* center, int32_t b, int32_t c, int32_t h,
                     int32_t w, int32_t crop_h, int32_t crop_w, int32_t border, float fill,
                     float* out) {
  const int ph = h + 2, pw = w + 2;
  for (int32_t s = 0; s < b; ++s) {
    /* utils.py:597-609 */
    const float ccx = center[s * 2 + 0] + 1.0f, ccy = center[s * 2 + 1] + 1.0f;
    const float center_x = ccx - (float)(pw / 2.0);
    const float center_y = ccy - (float)(ph / 2.0);
    for (int i = 0; i < crop_h; ++i)
      for (int j = 0; j < crop_w; ++j) {
        const float gx = ((float)j - (float)(crop_w / 2.0) + center_x) / (float)(pw / 2.0);
        const float gy = ((float)i - (float)(crop_h / 2.0) + center_y) / (float)(ph / 2.0);
        /* ATen GridSamplerKernel.cpp ComputeLocation<align_corners=true>:
         * unnormalize(in) = (in + 1) * ((size - 1) / 2) */
        float ix = (gx + 1.0f) * ((float)(pw - 1) / 2.0f);
        float iy = (gy + 1.0f) * ((float)(ph - 1) / 2.0f);
        if (border) {
          ix = fminf((float)(pw - 1), fmaxf(ix, 0.0f));
          iy = fminf((float)(ph - 1), fmaxf(iy, 0.0f));
        }
        const float rx = nearbyintf(ix), ry = nearbyintf(iy);
        const int inb = (rx >= 0.0f) & (rx < (float)pw) & (ry >= 0.0f) & (ry < (float)ph);
        for (int ch = 0; ch < c; ++ch) {
          float v = 0.0f;
          if (inb) {
            const int X = (int)rx, Y = (int)ry;
            if (X >= 1 && X <= w && Y >= 1 && Y <= h)
              v = image[(((int64_t)s * c + ch) * h + (Y - 1)) * w + (X - 1)];
            else
              v = fill; /* the constant pad ring */
          }
          out[(((int64_t)s * c + ch) * crop_h + i) * crop_w + j] = v;
        }
      }
  }
  return 0;
}

int dmo_max_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}
