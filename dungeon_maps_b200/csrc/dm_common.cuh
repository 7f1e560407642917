// Shared device-side pieces of the dungeon_maps_b200 kernels (sm_100a).
//
// Numerics contract (DESIGN.md "Numerics"): every reference torch op is one IEEE
// float32 rounding.  All coordinate math below is written with the __f*_rn
// intrinsics, which nvcc never contracts into FMAs (the files are additionally
// compiled with --fmad=false); __fmaf_rn appears only where the reference's
// sgemm fused (utils.py:329 → at::bmm → MKL, see DmStep in the public header).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dungeon_maps_b200.h"

namespace dm {

// ---- tracing: NVTX ranges around every C entry point (SURVEY.md §5) ---------------------------------------------
// NVTX v3 is header-only and resolves its injection library at run time: no link dependency, and a push / pop pair
// costs a few nanoseconds when no tool is attached.  nsys / ncu --nvtx then show `dm_orth_project_f32`, `dm_builder_merge`
// ... as ranges on the calling thread with the kernels they queued underneath.
#include <nvtx3/nvToolsExt.h>
struct DmRange {
  explicit DmRange(const char* name) { nvtxRangePushA(name); }
  ~DmRange() { nvtxRangePop(); }
  DmRange(const DmRange&) = delete;
  DmRange& operator=(const DmRange&) = delete;
};
#define DM_TRACE() ::DmRange dm_range_(__func__)

// ---- launch accounting / error plumbing -------------------------------------
extern int64_t g_launches;  // defined in dm_api.cu

#define DM_CUDA_OK(expr)                                  \
  do {                                                    \
    cudaError_t _e = (expr);                              \
    if (_e != cudaSuccess) return static_cast<int>(_e);   \
  } while (0)

#define DM_LAUNCHED()                                     \
  do {                                                    \
    ++::dm::g_launches;                                   \
    cudaError_t _e = cudaPeekAtLastError();               \
    if (_e != cudaSuccess) return static_cast<int>(_e);   \
  } while (0)

// SM count of the current device (148 on a B200), queried once per device: grids are sized in multiples of it.
int sm_count();  // dm_api.cu

// ---- host-side parameter packing (dm_params.cu) --------------------------------------------------
void yaw_matrix(const DmPoseCfg& c, float yaw, float sin_yaw, float cos_yaw, float* R);  // utils.py:318-327, axis (0, 1, 0)
void put_step(float* words, int kind, const float* R, const float* t, int fused);
bool local_step_is_fast(const DmPoseCfg& c);  // the pitch step has the structure DmProjCfg.fast_steps >= 1 promises
bool yaw_step_is_fast(const float* R);

// ---- ordered scatter-reduce for sum / mean / prod (dm_ordered.cu) ---------------------------------
// keys[i] = output cell of point i (or ~0: dropped), consumed; values[i]; canvas holds the starting values and
// receives the cells folded in ascending point index (the reference's CPU order).  n < 2^31.
// mask_or (optional): set to 1 where the fold changed the cell (utils.py:489-491).
int ordered_reduce(unsigned long long* keys, const float* values, long long n, int key_bits, int reduction,
                   float* canvas, uint8_t* mask_or, cudaStream_t stream);
int bits_for(unsigned long long max_key_exclusive);

// dm_fuse_scatter_track_f32 with `prefilled`: the canvases already hold the fill (dm_fuse.cu; used by dm_builder.cu)
int fuse_scatter_track(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C, const DmFuseTarget* target,
                       float* topdown, uint8_t* mask, float* height, int64_t* next_bbox, int32_t* next_plane_box,
                       int prefilled, void* stream);

// MapBuilder.plot fused with pass 1 of the merge (dm_builder.cu): the depth-only projection writes its key planes
// (dm_project.cu: hmap_project_keys, at most 64 frames, DM_EINVAL otherwise / when the height-map path is switched off),
// and ONE kernel resolves them into the local map and reduces that map's contribution to the merge's bounding box
// (dm_fuse.cu: hmap_resolve_with_bbox) — instead of resolve, bbox init and a bbox kernel that scans the mask just written.
int hmap_project_keys(const float* depth, const uint8_t* valid, const DmProjSample* samples, const DmProjCfg* cfg,
                      int32_t b, void* workspace, size_t workspace_bytes, cudaStream_t stream, uint32_t** planes,
                      unsigned long long* slot_words);
int hmap_resolve_with_bbox(uint32_t* planes, unsigned long long slot_words, const DmProjCfg* cfg, int32_t b,
                           float* topdown, uint8_t* mask, const DmFuseSource* local, float target_res,
                           const int64_t* seed, int64_t* bbox, cudaStream_t stream);
// pass 1 over `sources` into an ALREADY initialised bbox (dm_fuse.cu)
int fuse_bbox_accumulate(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C, float target_res,
                         int64_t* bbox, cudaStream_t stream);

// ---- reference arithmetic ------------------------------------------------------
struct V3 {
  float x, y, z;
};

// utils.py:329 (see DmStep: fused = MKL sgemm FMA chain, otherwise ATen's naive loop).
__device__ __forceinline__ V3 rot(const float* __restrict__ R, V3 p, int fused) {
  V3 o;
  if (fused) {
    o.x = __fmaf_rn(R[6], p.z, __fmaf_rn(R[3], p.y, __fmul_rn(R[0], p.x)));
    o.y = __fmaf_rn(R[7], p.z, __fmaf_rn(R[4], p.y, __fmul_rn(R[1], p.x)));
    o.z = __fmaf_rn(R[8], p.z, __fmaf_rn(R[5], p.y, __fmul_rn(R[2], p.x)));
  } else {
    o.x = __fadd_rn(__fadd_rn(__fmul_rn(R[0], p.x), __fmul_rn(R[3], p.y)), __fmul_rn(R[6], p.z));
    o.y = __fadd_rn(__fadd_rn(__fmul_rn(R[1], p.x), __fmul_rn(R[4], p.y)), __fmul_rn(R[7], p.z));
    o.z = __fadd_rn(__fadd_rn(__fmul_rn(R[2], p.x), __fmul_rn(R[5], p.y)), __fmul_rn(R[8], p.z));
  }
  return o;
}

// utils.py:229-259: all three components are added (the zeros too).
__device__ __forceinline__ V3 add3(V3 p, const float* __restrict__ t) {
  return V3{__fadd_rn(p.x, t[0]), __fadd_rn(p.y, t[1]), __fadd_rn(p.z, t[2])};
}

// maps.py:753-942.
__device__ __forceinline__ V3 apply_step(const DmStep& s, V3 p) {
  if (s.kind == DM_STEP_ROT_THEN_ADD) return add3(rot(s.R, p, s.fused), s.t);
  if (s.kind == DM_STEP_ADD_THEN_ROT) return rot(s.R, add3(p, s.t), s.fused);
  if (s.kind == DM_STEP_ADD) return add3(p, s.t);
  if (s.kind == DM_STEP_ROT) return rot(s.R, p, s.fused);
  return p;
}

// maps.py:667-679 image_to_camera_space for pixel (row r, col c).
__device__ __forceinline__ V3 unproject(int r, int c, float z, int H, float fx, float fy, float cx,
                                        float cy, int flip_h) {
  const float yy = flip_h ? __fsub_rn((float)(H - 1), (float)r) : (float)r;
  V3 p;
  p.x = __fmul_rn(__fdiv_rn(__fsub_rn((float)c, cx), fx), z);
  p.y = __fmul_rn(__fdiv_rn(__fsub_rn(yy, cy), fy), z);
  p.z = z;
  return p;
}

// maps.py:1004-1013 map_quantize, kept in float: floor(x + 0.5) as an integral float.  The
// reference casts to int64 (NaN / out of range → INT64_MIN on x86) and bounds-checks after;
// comparing the float against [0, size) gives the same verdict for every input.
__device__ __forceinline__ void quantize_f(float x, float z, float woff, float hoff, float res,
                                           int Mh, int flip_h, float* xf, float* zf) {
  const float xb = __fadd_rn(__fdiv_rn(x, res), woff);
  float zb = __fadd_rn(__fdiv_rn(z, res), hoff);
  if (flip_h) zb = __fsub_rn((float)(Mh - 1), zb);
  *xf = floorf(__fadd_rn(xb, 0.5f));
  *zf = floorf(__fadd_rn(zb, 0.5f));
}

// maps.py:1021-1087 map_dequantize of the bins (xb, zb), given as floats.
__device__ __forceinline__ void dequantize_f(float xb, float zb, float woff, float hoff, float res, int Mh,
                                             int flip_h, float* x, float* z) {
  if (flip_h) zb = __fsub_rn((float)(Mh - 1), zb);  // maps.py:1081-1084
  *z = __fmul_rn(__fsub_rn(zb, hoff), res);
  *x = __fmul_rn(__fsub_rn(xb, woff), res);
}

// Tensor.to(int64) on x86: cvttss2si semantics.
__device__ __forceinline__ long long f2i64(float v) {
  if (!(v >= -9223372036854775808.0f && v < 9223372036854775808.0f)) return (long long)0x8000000000000000ULL;
  return (long long)v;
}

// ---- order-preserving keys ------------------------------------------------------
// enc() maps float order onto unsigned order; key 0 is reserved for "cell untouched" and is
// never produced for a value that passed the `better than fill` test.  A min-reduction
// stores ~enc() so that one atomicMax serves both.
__device__ __forceinline__ uint32_t enc(float v) {
  const uint32_t b = __float_as_uint(v);
  // negative: flip all bits; non-negative: set the sign bit  ==  b ^ (sign-extension | 0x80000000)
  return b ^ ((uint32_t)((int32_t)b >> 31) | 0x80000000u);
}
__device__ __forceinline__ float dec(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
__device__ __forceinline__ uint32_t enc_red(float v, int is_min) { return is_min ? ~enc(v) : enc(v); }
__device__ __forceinline__ float dec_red(uint32_t k, int is_min) { return dec(is_min ? ~k : k); }
// torch_scatter semantics: `src > out` (max) / `src < out` (min); NaN never wins.
__device__ __forceinline__ bool better(float v, float cur, int is_min) {
  return is_min ? (v < cur) : (v > cur);
}

// Raw-float atomic max/min on a canvas holding plain floats (no key decode needed):
// non-negative floats order like signed ints, negative floats order inversely as unsigned.
__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
  if (!(__float_as_uint(v) & 0x80000000u))
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else
    atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_min_f32(float* addr, float v) {
  if (!(__float_as_uint(v) & 0x80000000u))
    atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else
    atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

// ---- streaming memory access ------------------------------------------------------
// Inputs are read exactly once: bypass L1 allocation, mark evict-first in L2 so the
// accumulation ring (re-used every frame) keeps its L2 residency.
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f1(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream_f4(float* p, float4 v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void st_stream_f1(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void st_stream_f2(float* p, float a, float b) {
  asm volatile("st.global.cs.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void st_stream_u16(uint8_t* p, uint32_t v) {
  asm volatile("st.global.cs.u16 [%0], %1;" ::"l"(p), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ void st_stream_u32(void* p, uint32_t v) {
  asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_stream_u4(void* p, uint32_t v) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1,%1,%1,%1};" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_stream_u8(uint8_t* p, uint8_t v) {
  asm volatile("st.global.cs.u8 [%0], %1;" ::"l"(p), "r"((uint32_t)v) : "memory");
}

}  // namespace dm
