// Materialising primitives: the reference's public L0/L1 functions for callers that ask for
// the intermediate tensors (TopdownMap.get_coords/get_points, user code).  Each is one
// element-wise (or scatter) kernel with the reference's float32 op order.
//   utils.rotate / utils.translate          utils.py:229-330
//   camera/local/global space transforms    maps.py:753-942
//   image_to_camera_space / camera_to_image maps.py:616-751
//   depth_map_to_point_cloud                maps.py:462-545
//   map_quantize / map_dequantize           maps.py:944-1087
//   scatter_tensor / project (2-D canvas)   utils.py:389-492, maps.py:1089-1173
//   crop_topdown_map                        maps.py:1959-2037, utils.py:571-652
#include "dm_common.cuh"

namespace dm {

constexpr int kThreads = 256;

static bool aligned_to(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

static unsigned grid_for(long long items) {
  long long blocks = (items + kThreads - 1) / kThreads;
  const long long cap = (long long)sm_count() * 8 * 2;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

#define DM_GRID_STRIDE(i, n) \
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (long long)gridDim.x * blockDim.x)

// xyz point clouds are arrays of structures (n, 3): a thread takes FOUR consecutive points = 48 bytes = three
// 128-bit accesses (the warp reads / writes 1.5 KB contiguous per instruction triple) instead of 3 stride-3 scalar
// accesses per point, which left two thirds of every sector to the L1 (round 1).  `vec`: both arrays 16-byte aligned.
struct P4 {
  float v[12];
};
__device__ __forceinline__ P4 load_p4(const float* __restrict__ pts, long long i0, long long total, bool vec) {
  P4 q;
  if (vec && i0 + 3 < total) {
    const float4* s4 = reinterpret_cast<const float4*>(pts + i0 * 3);
    const float4 a = __ldg(s4), b = __ldg(s4 + 1), c = __ldg(s4 + 2);
    q.v[0] = a.x; q.v[1] = a.y; q.v[2] = a.z; q.v[3] = a.w; q.v[4] = b.x; q.v[5] = b.y; q.v[6] = b.z; q.v[7] = b.w;
    q.v[8] = c.x; q.v[9] = c.y; q.v[10] = c.z; q.v[11] = c.w;
  } else {
#pragma unroll
    for (int k = 0; k < 12; ++k) q.v[k] = (i0 * 3 + k < total * 3) ? pts[i0 * 3 + k] : 0.0f;
  }
  return q;
}
__device__ __forceinline__ void store_p4(float* __restrict__ out, long long i0, long long total, bool vec, const P4& q) {
  if (vec && i0 + 3 < total) {
    float4* d4 = reinterpret_cast<float4*>(out + i0 * 3);
    d4[0] = make_float4(q.v[0], q.v[1], q.v[2], q.v[3]);
    d4[1] = make_float4(q.v[4], q.v[5], q.v[6], q.v[7]);
    d4[2] = make_float4(q.v[8], q.v[9], q.v[10], q.v[11]);
  } else {
#pragma unroll
    for (int k = 0; k < 12; ++k)
      if (i0 * 3 + k < total * 3) out[i0 * 3 + k] = q.v[k];
  }
}

__global__ void __launch_bounds__(kThreads)
transform_points_kernel(const float* __restrict__ pts, const DmStep* __restrict__ steps, int n_steps,
                        long long n, long long total, float* __restrict__ out, int vec) {
  DM_GRID_STRIDE(g, (total + 3) / 4) {
    const long long i0 = g * 4;
    P4 q = load_p4(pts, i0, total, vec);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (i0 + j >= total) break;
      const int s = (int)((i0 + j) / n);
      V3 p{q.v[3 * j], q.v[3 * j + 1], q.v[3 * j + 2]};
      for (int k = 0; k < n_steps; ++k) p = apply_step(steps[s * n_steps + k], p);
      q.v[3 * j] = p.x; q.v[3 * j + 1] = p.y; q.v[3 * j + 2] = p.z;
    }
    store_p4(out, i0, total, vec, q);
  }
}

__global__ void __launch_bounds__(kThreads)
image_camera_kernel(const float* __restrict__ pts, long long n, float fx, float fy, float cx, float cy,
                    int flip_h, int height, int to_image, float* __restrict__ out, int vec) {
  DM_GRID_STRIDE(g, (n + 3) / 4) {
    const long long i0 = g * 4;
    P4 q = load_p4(pts, i0, n, vec);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float x = q.v[3 * j], y = q.v[3 * j + 1];
      const float z = q.v[3 * j + 2];
      if (!to_image) {  // maps.py:670-678
        if (flip_h) y = __fsub_rn((float)(height - 1), y);
        x = __fmul_rn(__fdiv_rn(__fsub_rn(x, cx), fx), z);
        y = __fmul_rn(__fdiv_rn(__fsub_rn(y, cy), fy), z);
      } else {  // maps.py:743-747
        const float ze = __fadd_rn(z, 1e-7f);
        x = __fadd_rn(__fmul_rn(__fdiv_rn(x, ze), fx), cx);
        y = __fadd_rn(__fmul_rn(__fdiv_rn(y, ze), fy), cy);
        if (flip_h) y = __fsub_rn((float)(height - 1), y);
      }
      q.v[3 * j] = x; q.v[3 * j + 1] = y;
    }
    store_p4(out, i0, n, vec, q);
  }
}

// four consecutive pixels per thread: one 128-bit depth load, three 128-bit point stores, one 32-bit valid store
__global__ void __launch_bounds__(kThreads)
depth_to_points_kernel(const float* __restrict__ depth, const uint8_t* __restrict__ valid_in, long long total,
                       int H, int W, float fx, float fy, float cx, float cy, int flip_h, int has_tmin,
                       float tmin, int has_tmax, float tmax, float* __restrict__ pts,
                       uint8_t* __restrict__ valid_out, int vec) {
  const int N = H * W;
  DM_GRID_STRIDE(g, (total + 3) / 4) {
    const long long i0 = g * 4;
    const bool full = vec && i0 + 3 < total;
    float z[4];
    uint32_t vin = 0x01010101u;
    if (full) {
      const float4 z4 = ld_stream_f4(depth + i0);
      z[0] = z4.x; z[1] = z4.y; z[2] = z4.z; z[3] = z4.w;
      if (valid_in) vin = *reinterpret_cast<const uint32_t*>(valid_in + i0);
    } else {
      vin = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        z[j] = i0 + j < total ? depth[i0 + j] : 0.0f;
        if (i0 + j < total && (!valid_in || valid_in[i0 + j])) vin |= 1u << (8 * j);
      }
    }
    int n = (int)(i0 % N);
    int r = n / W, c = n - r * W;
    P4 q;
    uint32_t vout = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const V3 p = unproject(r, c, z[j], H, fx, fy, cx, cy, flip_h);
      q.v[3 * j] = p.x; q.v[3 * j + 1] = p.y; q.v[3 * j + 2] = p.z;
      bool ok = ((vin >> (8 * j)) & 0xffu) != 0;
      if (has_tmax) ok = ok && (z[j] <= tmax);
      if (has_tmin) ok = ok && (z[j] >= tmin);
      vout |= (ok ? 1u : 0u) << (8 * j);
      if (++c == W) { c = 0; if (++r == H) r = 0; }
    }
    store_p4(pts, i0, total, vec, q);
    if (full) {
      *reinterpret_cast<uint32_t*>(valid_out + i0) = vout;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (i0 + j < total) valid_out[i0 + j] = (uint8_t)((vout >> (8 * j)) & 1u);
    }
  }
}

__global__ void __launch_bounds__(kThreads)
quantize_kernel(const float* __restrict__ x, const float* __restrict__ z, const float* __restrict__ woff,
                const float* __restrict__ hoff, long long n, long long total, float res, int Mh, int flip_h,
                long long* __restrict__ xb, long long* __restrict__ zb) {
  DM_GRID_STRIDE(i, total) {
    const int s = (int)(i / n);
    float xf, zf;
    quantize_f(x[i], z[i], woff[s], hoff[s], res, Mh, flip_h, &xf, &zf);
    xb[i] = f2i64(xf);
    zb[i] = f2i64(zf);
  }
}

__global__ void __launch_bounds__(kThreads)
dequantize_kernel(const float* __restrict__ xb, const float* __restrict__ zb, const float* __restrict__ woff,
                  const float* __restrict__ hoff, long long n, long long total, float res, int Mh, int flip_h,
                  float* __restrict__ x, float* __restrict__ z) {
  DM_GRID_STRIDE(i, total) {
    const int s = (int)(i / n);
    dequantize_f(xb[i], zb[i], woff[s], hoff[s], res, Mh, flip_h, &x[i], &z[i]);
  }
}

__global__ void __launch_bounds__(kThreads)
fill_kernel(float* __restrict__ a, long long n, float v) {
  DM_GRID_STRIDE(i, n) a[i] = v;
}

__global__ void __launch_bounds__(kThreads)
copy_kernel(const float* __restrict__ a, float* __restrict__ b, long long n) {
  DM_GRID_STRIDE(i, n) b[i] = a[i];
}

// reduction: 0 max, 1 min (torch_scatter: `src > out` / `src < out`, NaN never wins): order-independent atomics.
__global__ void __launch_bounds__(kThreads)
scatter_kernel(const float* __restrict__ values, const long long* __restrict__ coords,
               const uint8_t* __restrict__ valid, long long N, long long total, int Mh, int Mw, int reduction,
               float* __restrict__ canvas) {
  const long long M = (long long)Mh * Mw;
  DM_GRID_STRIDE(i, total) {
    if (valid && !valid[i]) continue;
    const long long r = coords[i * 2], c = coords[i * 2 + 1];
    if (r < 0 || r >= Mh || c < 0 || c >= Mw) continue;  // utils.py:448-453
    const float v = values[i];
    if (v != v) continue;
    float* dst = canvas + ((i / N) * M + r * Mw + c);
    if (reduction) atomic_min_f32(dst, v); else atomic_max_f32(dst, v);
  }
}

// 2 sum, 3 mean, 4 prod (utils.py:70-76) depend on the order of the hits: the points get the key of their cell and
// dm_ordered.cu folds them in the reference's index order (bit-identical, deterministic).
__global__ void __launch_bounds__(kThreads)
scatter_keys_kernel(const long long* __restrict__ coords, const uint8_t* __restrict__ valid, long long N,
                    long long total, int Mh, int Mw, unsigned long long* __restrict__ keys) {
  const long long M = (long long)Mh * Mw;
  DM_GRID_STRIDE(i, total) {
    unsigned long long k = ~0ull;
    const long long r = coords[i * 2], c = coords[i * 2 + 1];
    if ((!valid || valid[i]) && r >= 0 && r < Mh && c >= 0 && c < Mw) k = (unsigned long long)((i / N) * M + r * Mw + c);
    keys[i] = k;
  }
}

__global__ void __launch_bounds__(kThreads)
changed_fill_kernel(const float* __restrict__ now, float fill, long long n, uint8_t* __restrict__ mask) {
  DM_GRID_STRIDE(i, n) {
    float d = fabsf(__fsub_rn(now[i], fill));
    if (d != d) d = 0.0f;
    mask[i] = d != 0.0f;
  }
}

// utils.py:489-491 with an arbitrary "before" canvas.
__global__ void __launch_bounds__(kThreads)
changed_kernel(const float* __restrict__ now, const float* __restrict__ before, long long n,
               uint8_t* __restrict__ mask) {
  DM_GRID_STRIDE(i, n) {
    float d = fabsf(__fsub_rn(now[i], before[i]));
    if (d != d) d = 0.0f;
    mask[i] = d != 0.0f;
  }
}

// generate_crop_grid (utils.py:597-609) + grid_sample(nearest, align_corners=True) on the image
// padded by one ring of `fill` (utils.py:639-650).  Source index as ATen's CPU kernel computes it:
// unnormalize(g) = (g + 1) * ((size - 1) / 2); border mode clamps before rounding; nearbyint.
template <typename T>
__global__ void __launch_bounds__(kThreads)
crop_kernel(const T* __restrict__ image, const float* __restrict__ center, int b, int c, int h, int w, int ch_,
            int cw_, int border, T fill, T zero, T* __restrict__ out) {
  const int ph = h + 2, pw = w + 2;
  const long long per = (long long)ch_ * cw_;
  const long long total = (long long)b * c * per;
  const float half_pw = (float)(pw / 2.0), half_ph = (float)(ph / 2.0);
  const float half_cw = (float)(cw_ / 2.0), half_ch = (float)(ch_ / 2.0);
  DM_GRID_STRIDE(i, total) {
    const long long sc = i / per;
    const int o = (int)(i - sc * per);
    const int s = (int)(sc / c);
    const int oi = o / cw_, oj = o - oi * cw_;
    const float center_x = __fsub_rn(__fadd_rn(center[s * 2 + 0], 1.0f), half_pw);
    const float center_y = __fsub_rn(__fadd_rn(center[s * 2 + 1], 1.0f), half_ph);
    const float gx = __fdiv_rn(__fadd_rn(__fsub_rn((float)oj, half_cw), center_x), half_pw);
    const float gy = __fdiv_rn(__fadd_rn(__fsub_rn((float)oi, half_ch), center_y), half_ph);
    float ix = __fmul_rn(__fadd_rn(gx, 1.0f), __fdiv_rn((float)(pw - 1), 2.0f));
    float iy = __fmul_rn(__fadd_rn(gy, 1.0f), __fdiv_rn((float)(ph - 1), 2.0f));
    if (border) {
      ix = fminf((float)(pw - 1), fmaxf(ix, 0.0f));
      iy = fminf((float)(ph - 1), fmaxf(iy, 0.0f));
    }
    const float rx = nearbyintf(ix), ry = nearbyintf(iy);
    T v = zero;
    if (rx >= 0.0f && rx < (float)pw && ry >= 0.0f && ry < (float)ph) {
      const int X = (int)rx, Y = (int)ry;
      v = (X >= 1 && X <= w && Y >= 1 && Y <= h) ? image[(sc * h + (Y - 1)) * w + (X - 1)] : fill;
    }
    out[i] = v;
  }
}

// TopdownMap.select_egocentric: cell (r, c) of sample s's crop_h x crop_w window is map_dequantize(c, r) with the
// window's offsets, local_to_global_space with the sample's pose, map_quantize with the source's offsets, and a read
// of the source there (the fills outside it).  One thread per (sample, cell): the coordinates once, then the C planes.
// samples: DM_EGO_SAMPLE_WORDS floats per sample, [DmStep | source woff, hoff | window woff, hoff].
// height: plane stride hplane (0: one plane shared by the C channels, written once), NULL for height maps.
__global__ void __launch_bounds__(kThreads)
crop_egocentric_kernel(const float* __restrict__ top, const float* __restrict__ height, long long hplane,
                       const uint8_t* __restrict__ mask, int b, int C, int Hs, int Ws, float res, int flip_h,
                       const float* __restrict__ samples, int ch_, int cw_, float fill, float* __restrict__ out_top,
                       float* __restrict__ out_height, uint8_t* __restrict__ out_mask) {
  const long long per = (long long)ch_ * cw_;
  const long long plane = (long long)Hs * Ws;
  const long long total = (long long)b * per;
  const int Ch = hplane ? C : 1;  // height planes per sample, in and out
  DM_GRID_STRIDE(i, total) {
    const int s = (int)(i / per);
    const int o = (int)(i - s * per);
    const int r = o / cw_, c = o - r * cw_;
    const float* w = samples + (long long)s * DM_EGO_SAMPLE_WORDS;
    float lx, lz;
    dequantize_f((float)c, (float)r, w[18], w[19], res, ch_, flip_h, &lx, &lz);
    const V3 g = apply_step(*reinterpret_cast<const DmStep*>(w), V3{lx, 0.0f, lz});
    float xf, zf;
    quantize_f(g.x, g.z, w[16], w[17], res, Hs, flip_h, &xf, &zf);
    const bool in = xf >= 0.0f && xf < (float)Ws && zf >= 0.0f && zf < (float)Hs;
    const long long cell = in ? (long long)zf * Ws + (long long)xf : 0;
    const long long src = (long long)s * C * plane + cell;
    const long long dst = (long long)s * C * per + o;
    for (int k = 0; k < C; ++k) {
      out_top[dst + k * per] = in ? top[src + k * plane] : fill;
      out_mask[dst + k * per] = in ? mask[src + k * plane] : (uint8_t)0;
    }
    if (out_height) {
      const long long hsrc = (long long)s * Ch * plane + cell;
      const long long hdst = (long long)s * Ch * per + o;
      for (int k = 0; k < Ch; ++k)
        out_height[hdst + k * per] = in ? height[hsrc + k * plane] : -INFINITY;
    }
  }
}

}  // namespace dm

using namespace dm;

extern "C" int dm_transform_points_f32(const float* points, const DmStep* steps, int32_t n_steps, int32_t b,
                                       int64_t n, float* out, void* stream) {
  DM_TRACE();
  if (b < 0 || n < 0 || n_steps < 0) return DM_EINVAL;
  const long long total = (long long)b * n;
  if (total == 0) return DM_OK;
  if (!points || !out || (n_steps > 0 && !steps)) return DM_EINVAL;
  transform_points_kernel<<<grid_for((total + 3) / 4), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      points, steps, n_steps, n, total, out, aligned_to(points, 16) && aligned_to(out, 16));
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_image_camera_f32(const float* points, int64_t n, float fx, float fy, float cx, float cy,
                                   int32_t flip_h, int32_t height, int32_t to_image, float* out, void* stream) {
  DM_TRACE();
  if (n < 0) return DM_EINVAL;
  if (n == 0) return DM_OK;
  if (!points || !out) return DM_EINVAL;
  image_camera_kernel<<<grid_for((n + 3) / 4), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      points, n, fx, fy, cx, cy, flip_h, height, to_image, out, aligned_to(points, 16) && aligned_to(out, 16));
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_depth_to_points_f32(const float* depth, const uint8_t* valid_in, int64_t frames, int32_t H,
                                      int32_t W, float fx, float fy, float cx, float cy, int32_t flip_h,
                                      int32_t has_tmin, float tmin, int32_t has_tmax, float tmax, float* points,
                                      uint8_t* valid_out, void* stream) {
  DM_TRACE();
  if (frames < 0 || H <= 0 || W <= 0) return DM_EINVAL;
  const long long total = (long long)frames * H * W;
  if (total == 0) return DM_OK;
  if (!depth || !points || !valid_out) return DM_EINVAL;
  depth_to_points_kernel<<<grid_for((total + 3) / 4), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      depth, valid_in, total, H, W, fx, fy, cx, cy, flip_h, has_tmin, tmin, has_tmax, tmax, points, valid_out,
      aligned_to(depth, 16) && aligned_to(points, 16) && aligned_to(valid_out, 4) && (!valid_in || aligned_to(valid_in, 4)));
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_map_quantize_f32(const float* x, const float* z, const float* width_offset,
                                   const float* height_offset, int32_t b, int64_t n, float map_res,
                                   int32_t map_height, int32_t flip_h, int64_t* x_bin, int64_t* z_bin,
                                   void* stream) {
  DM_TRACE();
  if (b < 0 || n < 0) return DM_EINVAL;
  const long long total = (long long)b * n;
  if (total == 0) return DM_OK;
  if (!x || !z || !width_offset || !height_offset || !x_bin || !z_bin) return DM_EINVAL;
  quantize_kernel<<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x, z, width_offset, height_offset, n, total, map_res, map_height, flip_h,
      reinterpret_cast<long long*>(x_bin), reinterpret_cast<long long*>(z_bin));
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_map_dequantize_f32(const float* x_bin, const float* z_bin, const float* width_offset,
                                     const float* height_offset, int32_t b, int64_t n, float map_res,
                                     int32_t map_height, int32_t flip_h, float* x, float* z, void* stream) {
  DM_TRACE();
  if (b < 0 || n < 0) return DM_EINVAL;
  const long long total = (long long)b * n;
  if (total == 0) return DM_OK;
  if (!x || !z || !width_offset || !height_offset || !x_bin || !z_bin) return DM_EINVAL;
  dequantize_kernel<<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x_bin, z_bin, width_offset, height_offset, n, total, map_res, map_height, flip_h, x, z);
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_scatter_f32(const float* values, const int64_t* coords, const uint8_t* valid, int64_t B,
                              int64_t N, int32_t Mh, int32_t Mw, int32_t has_fill, float fill_value,
                              int32_t reduction, const float* canvas_in, float* canvas_out, uint8_t* mask,
                              void* stream_) {
  DM_TRACE();
  if (B < 0 || N < 0 || Mh <= 0 || Mw <= 0 || reduction < 0 || reduction > 4) return DM_EINVAL;
  if (B == 0) return DM_OK;
  if (!canvas_out || !mask || (N > 0 && (!values || !coords))) return DM_EINVAL;
  if (!has_fill && !canvas_in) return DM_EINVAL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long n_out = (long long)B * Mh * Mw;
  if (has_fill)  // utils.py:472-473
    fill_kernel<<<grid_for(n_out), kThreads, 0, stream>>>(canvas_out, n_out, fill_value);
  else           // utils.py:467: the scatter works on a copy of the caller's canvas
    copy_kernel<<<grid_for(n_out), kThreads, 0, stream>>>(canvas_in, canvas_out, n_out);
  DM_LAUNCHED();
  const long long total = (long long)B * N;
  if (total > 0 && reduction < 2) {
    scatter_kernel<<<grid_for(total), kThreads, 0, stream>>>(values, reinterpret_cast<const long long*>(coords),
                                                             valid, N, total, Mh, Mw, reduction, canvas_out);
    DM_LAUNCHED();
  } else if (total > 0) {
    if (total >= (1ll << 31)) return DM_EINVAL;
    unsigned long long* keys = nullptr;  // stream-ordered scratch
    DM_CUDA_OK(cudaMallocAsync(&keys, (size_t)total * 8, stream));
    scatter_keys_kernel<<<grid_for(total), kThreads, 0, stream>>>(reinterpret_cast<const long long*>(coords), valid, N,
                                                                  total, Mh, Mw, keys);
    DM_LAUNCHED();
    const int rc = ordered_reduce(keys, values, total, bits_for((unsigned long long)n_out), reduction, canvas_out, nullptr, stream);
    DM_CUDA_OK(cudaFreeAsync(keys, stream));
    if (rc != DM_OK) return rc;
  }
  if (has_fill)
    changed_fill_kernel<<<grid_for(n_out), kThreads, 0, stream>>>(canvas_out, fill_value, n_out, mask);
  else
    changed_kernel<<<grid_for(n_out), kThreads, 0, stream>>>(canvas_out, canvas_in, n_out, mask);
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_crop_nearest_f32(const float* image, const float* center, int32_t b, int32_t c, int32_t h,
                                   int32_t w, int32_t crop_h, int32_t crop_w, int32_t border, float fill,
                                   float* out, void* stream) {
  DM_TRACE();
  if (b < 0 || c < 0 || h <= 0 || w <= 0 || crop_h < 0 || crop_w < 0) return DM_EINVAL;
  const long long total = (long long)b * c * crop_h * crop_w;
  if (total == 0) return DM_OK;
  if (!image || !center || !out) return DM_EINVAL;
  crop_kernel<float><<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      image, center, b, c, h, w, crop_h, crop_w, border, fill, 0.0f, out);
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_crop_nearest_u8(const uint8_t* image, const float* center, int32_t b, int32_t c, int32_t h,
                                  int32_t w, int32_t crop_h, int32_t crop_w, uint8_t* out, void* stream) {
  DM_TRACE();
  if (b < 0 || c < 0 || h <= 0 || w <= 0 || crop_h < 0 || crop_w < 0) return DM_EINVAL;
  const long long total = (long long)b * c * crop_h * crop_w;
  if (total == 0) return DM_OK;
  if (!image || !center || !out) return DM_EINVAL;
  // the reference crops masks with fill_value=False → border mode over a ring of zeros
  crop_kernel<uint8_t><<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      image, center, b, c, h, w, crop_h, crop_w, 1, (uint8_t)0, (uint8_t)0, out);
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_crop_egocentric_f32(const float* topdown, const float* height, int64_t height_plane_stride,
                                      const uint8_t* mask, int32_t b, int32_t C, int32_t Hs, int32_t Ws, float map_res,
                                      int32_t flip_h, const float* samples, int32_t crop_h, int32_t crop_w,
                                      float fill_value, float* out_topdown, float* out_height, uint8_t* out_mask,
                                      void* stream) {
  DM_TRACE();
  if (b <= 0 || C <= 0 || Hs <= 0 || Ws <= 0 || crop_h <= 0 || crop_w <= 0 || !(map_res > 0.0f)) return DM_EINVAL;
  if ((long long)crop_h * crop_w >= (1ll << 31) || (long long)Hs * Ws >= (1ll << 31)) return DM_EINVAL;
  if (!topdown || !mask || !samples || !out_topdown || !out_mask) return DM_EINVAL;
  if (!height != !out_height) return DM_EINVAL;
  if (height && height_plane_stride != 0 && height_plane_stride != (int64_t)Hs * Ws) return DM_EINVAL;
  if (!aligned_to(samples, 4)) return DM_EINVAL;
  const long long total = (long long)b * crop_h * crop_w;
  crop_egocentric_kernel<<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      topdown, height, height ? height_plane_stride : 0, mask, b, C, Hs, Ws, map_res, flip_h, samples, crop_h, crop_w,
      fill_value, out_topdown, out_height, out_mask);
  DM_LAUNCHED();
  return DM_OK;
}
