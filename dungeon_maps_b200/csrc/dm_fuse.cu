// MapBuilder merge: fuse_topdown_maps, /root/reference/dungeon_maps/maps.py:2181-2287.
//
// The reference turns every cell of every source map back into a 3-D point
// (height_map_to_point_cloud / map_dequantize, maps.py:547-612, 1021-1087), moves it into the
// target frame (maps.py:2059-2060, 2116-2117), takes ONE bounding box over all valid points of
// all samples and channels to size a fresh canvas (maps.py:2146-2179, host sync), re-quantises
// and scatter-maxes (maps.py:2232-2272).  Here that is two fused passes over the source cells,
// neither of which materialises a point: pass 1 reduces the bounding box, pass 2 scatters.
// Both passes give a block ONE plane (sample, channel) of ONE source at a time, so the sample's two
// transform steps and offsets sit in shared memory and all index arithmetic is 32-bit; a kernel is
// launched per source (at most 8).
#include "dm_common.cuh"

namespace dm {

constexpr int kFuseThreads = 256;
// block size of the two scanning passes (bbox, scatter): a block lives as long as its slowest warp, and the valid cells
// of a plane sit in one corner (config 4, µs per merge of all fuse kernels: 256 threads 343, 128: 323, 64: 334, 32: 349)
constexpr int kScanThreads = 128;
constexpr int kMaxSources = 8;
constexpr int kGroup = 16;  // mask bytes examined per work item (one 128-bit load)
#ifndef DM_FUSE_MIN_CELLS
#define DM_FUSE_MIN_CELLS 8192
#endif
constexpr long long kMinCellsPerBlock = DM_FUSE_MIN_CELLS;  // plane_grid: at least this many cells of a plane per block
int g_dense_shift = 1;      // test hook (dm_debug_set_dense_shift): 0 keeps every plane on the per-cell path

// Block-uniform state of the plane (one (sample, channel) image of one source) a block is scanning.
struct PlaneCtx {
  DmStep step0, step1;  // source local→global, global→target local (kind 0: none)
  float woff, hoff;
};

// Walks the valid cells of plane `plane` of `src`.  A lane examines kAhead groups of 16 mask bytes per round (aligned
// 128-bit loads, all in flight before the first is looked at), the warp then shares the valid cells it found evenly:
// cell number i of the round goes to lane i % 32, whichever lane's group it came from.  World maps are sparse — a
// grown config-4 canvas has ~5 valid cells per 512 examined, and even inside the explored corner they are outlines,
// not areas — so visiting a lane's own cells one after the other ran the ~150-instruction visitor with 4 of 32 lanes
// active on average (ncu r01k: 10.7 active threads per instruction, 75 M warp instructions for 1.5 M cells).
// visit(cell index in the plane, row, col) is instantiated once and reached by the whole warp together.
__device__ __forceinline__ uint32_t bits_of(const uint4 v) {
  const uint32_t m[4] = {v.x, v.y, v.z, v.w};
  uint32_t bits = 0;
#pragma unroll
  for (int j = 0; j < kGroup; ++j) bits |= ((m[j >> 2] >> ((j & 3) * 8)) & 0xffu) ? (1u << j) : 0u;
  return bits;
}

// The same walk restricted to the plane's bounding box of valid cells (rows r0..r1, columns c0..c1), as the scatter
// pass that wrote the map tracked it (DmFuseSource.plane_box).  A grown world map is mostly empty canvas: every
// environment's explored region is a small rectangle of the batch-wide canvas, and scanning the whole 155 MB of masks
// to find it again was the largest merge kernel after the fill (ncu r01m: 90 us at 25 % DRAM throughput).  Work item =
// (row of the box, 16-byte group of that row's column range); groups stay aligned to the plane's 16-byte grid, so a
// group may reach outside the box — where the mask is zero by construction.
template <typename F>
__device__ __forceinline__ void for_valid_cells_of_box(const DmFuseSource& src, long long plane, int r0, int r1, int c0,
                                                       int c1, F&& visit) {
  constexpr int kAhead = 4;
  if (r1 < r0 || c1 < c0) return;  // no valid cell in this plane
  const int n = src.h * src.w, w = src.w;
  const uint8_t* base = src.mask + plane * n;
  const int a0 = (int)(reinterpret_cast<uintptr_t>(base) & 15);
  const int gpr = ((c1 - c0 + 15) >> 4) + 1;            // groups per row, upper bound
  const long long items = (long long)(r1 - r0 + 1) * gpr;
  const int stride = gridDim.x * kScanThreads;
  const int lane = threadIdx.x & 31;
  auto group_offset = [&](long long item) -> int {       // plane-relative byte offset of the item's group, or INT_MIN
    if (item >= items) return INT_MIN;
    const int ri = (int)(item / gpr), gi = (int)(item - (long long)ri * gpr);
    const int r = r0 + ri;
    const int g = ((r * w + c0 + a0) >> 4) + gi;
    if (g > ((r * w + c1 + a0) >> 4)) return INT_MIN;    // past the row's last group
    if (ri > 0 && g <= (((r - 1) * w + c1 + a0) >> 4)) return INT_MIN;  // the previous row's item already took it
    return g * kGroup - a0;
  };
  for (long long iw = blockIdx.x * kScanThreads + (threadIdx.x & ~31); iw < items; iw += (long long)kAhead * stride) {
    int o[kAhead];
    uint4 v[kAhead];
#pragma unroll
    for (int k = 0; k < kAhead; ++k) {
      o[k] = group_offset(iw + lane + (long long)k * stride);
      v[k] = make_uint4(0u, 0u, 0u, 0u);
      if (o[k] != INT_MIN && o[k] >= 0 && o[k] + kGroup <= n) v[k] = __ldg(reinterpret_cast<const uint4*>(base + o[k]));
    }
    unsigned long long bits = 0;
#pragma unroll
    for (int k = 0; k < kAhead; ++k) {
      uint32_t bk = 0;
      if (o[k] != INT_MIN) {
        if (o[k] >= 0 && o[k] + kGroup <= n) {
          if (v[k].x | v[k].y | v[k].z | v[k].w) bk = bits_of(v[k]);
        } else {
          for (int j = 0; j < kGroup; ++j)
            if (o[k] + j >= 0 && o[k] + j < n && base[o[k] + j]) bk |= 1u << j;
        }
      }
      bits |= (unsigned long long)bk << (16 * k);
    }
    if (!__any_sync(0xffffffffu, bits != 0ull)) continue;
    const int cnt = __popcll(bits);
    int incl = cnt;
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, dd);
      if (lane >= dd) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t blo = (uint32_t)bits, bhi = (uint32_t)(bits >> 32);
    for (int first = 0; first < total; first += 32) {
      const int idx = first + lane;
      int L = 0;
#pragma unroll
      for (int step = 16; step >= 1; step >>= 1) {
        const int t = __shfl_sync(0xffffffffu, incl, L + step - 1);
        if (t <= idx) L += step;
      }
      L &= 31;
      const uint32_t lo_own = __shfl_sync(0xffffffffu, blo, L), hi_own = __shfl_sync(0xffffffffu, bhi, L);
      const int excl_own = __shfl_sync(0xffffffffu, incl - cnt, L);
      const int o0 = __shfl_sync(0xffffffffu, o[0], L), o1 = __shfl_sync(0xffffffffu, o[1], L);
      const int o2 = __shfl_sync(0xffffffffu, o[2], L), o3 = __shfl_sync(0xffffffffu, o[3], L);
      if (idx < total) {
        const int rank = idx - excl_own, nlo = __popc(lo_own);
        const int bit = rank < nlo ? (int)__fns(lo_own, 0, rank + 1) : 32 + (int)__fns(hi_own, 0, rank - nlo + 1);
        const int k = bit >> 4;
        const int cell = (k == 0 ? o0 : k == 1 ? o1 : k == 2 ? o2 : o3) + (bit & 15);
        const int r = cell / w;
        visit(cell, r, cell - r * w);
      }
    }
  }
}

template <typename F>
__device__ __forceinline__ void for_valid_cells_of_plane(const DmFuseSource& src, long long plane, F&& visit) {
  constexpr int kAhead = 4;  // groups per lane and round: 64 cells, one bit each in a 64-bit word
  const int n = src.h * src.w;
  const uint8_t* base = src.mask + plane * n;
  const int a0 = (int)(reinterpret_cast<uintptr_t>(base) & 15);  // bytes between the aligned-down start and the plane
  const int groups = (n + a0 + kGroup - 1) / kGroup;
  const int stride = gridDim.x * kScanThreads;
  const int lane = threadIdx.x & 31;
  // warp-uniform loop: gw is the group of lane 0
  for (int gw = blockIdx.x * kScanThreads + (threadIdx.x & ~31); gw < groups; gw += kAhead * stride) {
    const int g0 = gw + lane;
    uint4 v[kAhead];
#pragma unroll
    for (int k = 0; k < kAhead; ++k) {
      const int g = g0 + k * stride;
      const int o = g * kGroup - a0;  // plane-relative offset of the group's first byte (negative in the head group)
      v[k] = make_uint4(0u, 0u, 0u, 0u);
      if (g < groups && o >= 0 && o + kGroup <= n) v[k] = __ldg(reinterpret_cast<const uint4*>(base + o));
    }
    unsigned long long bits = 0;
#pragma unroll
    for (int k = 0; k < kAhead; ++k) {
      const int g = g0 + k * stride;
      const int o = g * kGroup - a0;
      uint32_t bk = 0;
      if (g < groups) {
        if (o >= 0 && o + kGroup <= n) {
          if (v[k].x | v[k].y | v[k].z | v[k].w) bk = bits_of(v[k]);
        } else {  // head / tail group of a plane whose start or size is not a multiple of 16: byte loads inside the plane
          for (int j = 0; j < kGroup; ++j)
            if (o + j >= 0 && o + j < n && base[o + j]) bk |= 1u << j;
        }
      }
      bits |= (unsigned long long)bk << (16 * k);
    }
    if (!__any_sync(0xffffffffu, bits != 0ull)) continue;
    // inclusive prefix sum of the lanes' cell counts
    const int cnt = __popcll(bits);
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t blo = (uint32_t)bits, bhi = (uint32_t)(bits >> 32);
    const int o0 = g0 * kGroup - a0;
    for (int first = 0; first < total; first += 32) {
      const int idx = first + lane;  // the cell of this round that is mine
      // owner = first lane whose inclusive count exceeds idx (binary search over the lanes)
      int L = 0;
#pragma unroll
      for (int step = 16; step >= 1; step >>= 1) {
        const int t = __shfl_sync(0xffffffffu, incl, L + step - 1);
        if (t <= idx) L += step;
      }
      L &= 31;  // idx >= total: any lane, result unused
      const int o_own = __shfl_sync(0xffffffffu, o0, L);
      const uint32_t lo_own = __shfl_sync(0xffffffffu, blo, L), hi_own = __shfl_sync(0xffffffffu, bhi, L);
      const int excl_own = __shfl_sync(0xffffffffu, incl - cnt, L);
      if (idx < total) {
        const int rank = idx - excl_own, nlo = __popc(lo_own);
        const int bit = rank < nlo ? (int)__fns(lo_own, 0, rank + 1) : 32 + (int)__fns(hi_own, 0, rank - nlo + 1);
        const int cell = o_own + (bit >> 4) * (stride * kGroup) + (bit & 15);
        const int r = cell / src.w;
        visit(cell, r, cell - r * src.w);
      }
    }
  }
}

// Walks the valid cells of a plane: inside its tracked bounding box when the source carries one, else all of it.
template <typename F>
__device__ __forceinline__ void for_valid_cells(const DmFuseSource& src, long long plane, F&& visit) {
  if (src.plane_box) {
    const int4 bx = __ldg(reinterpret_cast<const int4*>(src.plane_box) + plane);  // rmin, rmax, cmin, cmax
    const int r0 = max(bx.x, 0), r1 = min(bx.y, src.h - 1), c0 = max(bx.z, 0), c1 = min(bx.w, src.w - 1);
    for_valid_cells_of_box(src, plane, r0, r1, c0, c1, visit);
  } else {
    for_valid_cells_of_plane(src, plane, visit);
  }
}

// Loads the plane's sample parameters into shared memory (block-uniform), once per sample change.
__device__ __forceinline__ void load_plane_ctx(const DmFuseSource& src, int smp, PlaneCtx* ctx) {
  __syncthreads();
  if (threadIdx.x < 32) {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(src.steps + smp * 2);
    reinterpret_cast<uint32_t*>(&ctx->step0)[threadIdx.x] = s[threadIdx.x];  // 2 x 64 bytes = 32 words
  }
  if (threadIdx.x == 0) {
    ctx->woff = src.width_offset[smp];
    ctx->hoff = src.height_offset[smp];
  }
  __syncthreads();
}

// Point of source cell (row r, col c) of the plane, in the target frame.
__device__ __forceinline__ V3 source_point(const DmFuseSource& src, const PlaneCtx& ctx, const float* hplane, int cell,
                                           int r, int c) {
  // maps.py:1081-1086 map_dequantize
  float zb = (float)r;
  if (src.flip_h) zb = __fsub_rn((float)(src.h - 1), zb);
  V3 p;
  p.z = __fmul_rn(__fsub_rn(zb, ctx.hoff), src.map_res);
  p.x = __fmul_rn(__fsub_rn((float)c, ctx.woff), src.map_res);
  p.y = hplane[cell];
  if (ctx.step0.kind != DM_STEP_NONE) p = apply_step(ctx.step0, p);  // block-uniform branches
  if (ctx.step1.kind != DM_STEP_NONE) p = apply_step(ctx.step1, p);
  return p;
}

__global__ void fuse_bbox_init(long long* out, const long long* seed = nullptr) {
  if (seed) {  // start from a bounding box that an earlier scatter pass left for its output map
    for (int i = 0; i < 5; ++i) out[i] = seed[i];
    return;
  }
  out[0] = 0x7fffffffffffffffLL;          // min_x
  out[1] = (long long)0x8000000000000000ULL;  // max_x
  out[2] = 0x7fffffffffffffffLL;          // min_z
  out[3] = (long long)0x8000000000000000ULL;  // max_z
  out[4] = 0;                              // n_valid
}

// grid = (blocks per plane, planes folded into y)
__global__ void __launch_bounds__(kScanThreads, 1024 / kScanThreads)
fuse_bbox_kernel(const __grid_constant__ DmFuseSource src, int planes, int C, float res, long long* __restrict__ out) {
  __shared__ PlaneCtx ctx;
  long long mnx = 0x7fffffffffffffffLL, mxx = (long long)0x8000000000000000ULL;
  long long mnz = mnx, mxz = mxx;
  unsigned long long cnt = 0;
  int loaded = -1;
  for (int plane = blockIdx.y; plane < planes; plane += gridDim.y) {
    const int smp = plane / C, ch = plane - smp * C;
    if (smp != loaded) { load_plane_ctx(src, smp, &ctx); loaded = smp; }
    const float* hplane = src.height + (long long)smp * src.height_bstride + (long long)ch * src.height_cstride;
    for_valid_cells(src, plane, [&](int cell, int r, int c) {
      const V3 p = source_point(src, ctx, hplane, cell, r, c);
      // maps.py:2159-2165: map_quantize(width_offset=0., height_offset=0., flip_h=False)
      float xf, zf;
      quantize_f(p.x, p.z, 0.0f, 0.0f, res, 0, 0, &xf, &zf);
      const long long xi = f2i64(xf), zi = f2i64(zf);
      mnx = xi < mnx ? xi : mnx; mxx = xi > mxx ? xi : mxx;
      mnz = zi < mnz ? zi : mnz; mxz = zi > mxz ? zi : mxz;
      ++cnt;
    });
  }
  // warp then block reduction, one atomic per block per quantity
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const long long a = __shfl_xor_sync(0xffffffffu, mnx, o), b2 = __shfl_xor_sync(0xffffffffu, mxx, o);
    const long long c2 = __shfl_xor_sync(0xffffffffu, mnz, o), d2 = __shfl_xor_sync(0xffffffffu, mxz, o);
    const unsigned long long e2 = __shfl_xor_sync(0xffffffffu, cnt, o);
    mnx = a < mnx ? a : mnx; mxx = b2 > mxx ? b2 : mxx;
    mnz = c2 < mnz ? c2 : mnz; mxz = d2 > mxz ? d2 : mxz;
    cnt += e2;
  }
  __shared__ long long sm[kScanThreads / 32][4];
  __shared__ unsigned long long sc[kScanThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sm[warp][0] = mnx; sm[warp][1] = mxx; sm[warp][2] = mnz; sm[warp][3] = mxz; sc[warp] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kScanThreads / 32; ++w) {
      mnx = sm[w][0] < mnx ? sm[w][0] : mnx; mxx = sm[w][1] > mxx ? sm[w][1] : mxx;
      mnz = sm[w][2] < mnz ? sm[w][2] : mnz; mxz = sm[w][3] > mxz ? sm[w][3] : mxz;
      cnt += sc[w];
    }
    if (cnt) {
      atomicMin(out + 0, mnx); atomicMax(out + 1, mxx);
      atomicMin(out + 2, mnz); atomicMax(out + 3, mxz);
      atomicAdd(reinterpret_cast<unsigned long long*>(out + 4), cnt);
    }
  }
}

// MapBuilder.plot's resolve pass (dm_project.cu: hmap_resolve_kernel — key -> value / mask, plane zero again) fused
// with pass 1 of the merge over the map it writes: a cell that holds a key IS a valid cell of the local map, so its
// point goes through source_point() and quantize_f() right here (the operations of fuse_bbox_kernel, same bits) and
// the separate scan of the 5 MB of masks just written, its launch and the bbox init go away (20 + 4 us of a 292 us step).
__global__ void __launch_bounds__(256)
hmap_resolve_bbox_kernel(uint32_t* __restrict__ acc, unsigned long long slot_words, const DmProjCfg cfg, int vec,
                         float* __restrict__ topdown, uint8_t* __restrict__ mask,
                         const __grid_constant__ DmFuseSource src, float res, long long* __restrict__ out) {
  __shared__ PlaneCtx ctx;
  const int frame = blockIdx.y;
  load_plane_ctx(src, frame, &ctx);
  const int M = cfg.Mh * cfg.Mw;
  uint32_t* plane = acc + (size_t)frame * slot_words;
  float* tp = topdown + (size_t)frame * M;
  uint8_t* mp = mask + (size_t)frame * M;
  const float fill = cfg.fill_value;
  const int is_min = cfg.reduction;
  long long mnx = 0x7fffffffffffffffLL, mxx = (long long)0x8000000000000000ULL;
  long long mnz = mnx, mxz = mxx;
  unsigned long long cnt = 0;
  auto visit = [&](int m, float v) {  // valid cell m of the local map holding height v
    const int r = m / cfg.Mw, c = m - r * cfg.Mw;
    // maps.py:1081-1086 map_dequantize + the source's steps, exactly as source_point()
    float zb = (float)r;
    if (src.flip_h) zb = __fsub_rn((float)(src.h - 1), zb);
    V3 p;
    p.z = __fmul_rn(__fsub_rn(zb, ctx.hoff), src.map_res);
    p.x = __fmul_rn(__fsub_rn((float)c, ctx.woff), src.map_res);
    p.y = v;
    if (ctx.step0.kind != DM_STEP_NONE) p = apply_step(ctx.step0, p);
    if (ctx.step1.kind != DM_STEP_NONE) p = apply_step(ctx.step1, p);
    float xf, zf;  // maps.py:2159-2165: map_quantize(width_offset=0., height_offset=0., flip_h=False)
    quantize_f(p.x, p.z, 0.0f, 0.0f, res, 0, 0, &xf, &zf);
    const long long xi = f2i64(xf), zi = f2i64(zf);
    mnx = xi < mnx ? xi : mnx; mxx = xi > mxx ? xi : mxx;
    mnz = zi < mnz ? zi : mnz; mxz = zi > mxz ? zi : mxz;
    ++cnt;
  };
  for (int m0 = (blockIdx.x * 256 + threadIdx.x) * 4; m0 < M; m0 += gridDim.x * 1024) {
    if (vec && m0 + 3 < M) {
      const uint4 k = __ldcg(reinterpret_cast<const uint4*>(plane + m0));
      if (k.x | k.y | k.z | k.w) __stcg(reinterpret_cast<uint4*>(plane + m0), make_uint4(0u, 0u, 0u, 0u));
      const float v0 = k.x ? dec_red(k.x, is_min) : fill, v1 = k.y ? dec_red(k.y, is_min) : fill;
      const float v2 = k.z ? dec_red(k.z, is_min) : fill, v3 = k.w ? dec_red(k.w, is_min) : fill;
      st_stream_f4(tp + m0, make_float4(v0, v1, v2, v3));
      st_stream_u32(mp + m0, (k.x ? 1u : 0u) | (k.y ? 0x100u : 0u) | (k.z ? 0x10000u : 0u) | (k.w ? 0x1000000u : 0u));
      if (k.x) visit(m0, v0);
      if (k.y) visit(m0 + 1, v1);
      if (k.z) visit(m0 + 2, v2);
      if (k.w) visit(m0 + 3, v3);
    } else {
      for (int m = m0; m < min(m0 + 4, M); ++m) {
        const uint32_t k = __ldcg(plane + m);
        if (k) __stcg(plane + m, 0u);
        const float v = k ? dec_red(k, is_min) : fill;
        st_stream_f1(tp + m, v);
        st_stream_u8(mp + m, k ? 1 : 0);
        if (k) visit(m, v);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const long long a = __shfl_xor_sync(0xffffffffu, mnx, o), b2 = __shfl_xor_sync(0xffffffffu, mxx, o);
    const long long c2 = __shfl_xor_sync(0xffffffffu, mnz, o), d2 = __shfl_xor_sync(0xffffffffu, mxz, o);
    const unsigned long long e2 = __shfl_xor_sync(0xffffffffu, cnt, o);
    mnx = a < mnx ? a : mnx; mxx = b2 > mxx ? b2 : mxx;
    mnz = c2 < mnz ? c2 : mnz; mxz = d2 > mxz ? d2 : mxz;
    cnt += e2;
  }
  __shared__ long long sm[8][4];
  __shared__ unsigned long long sc[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sm[warp][0] = mnx; sm[warp][1] = mxx; sm[warp][2] = mnz; sm[warp][3] = mxz; sc[warp] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) {
      mnx = sm[w][0] < mnx ? sm[w][0] : mnx; mxx = sm[w][1] > mxx ? sm[w][1] : mxx;
      mnz = sm[w][2] < mnz ? sm[w][2] : mnz; mxz = sm[w][3] > mxz ? sm[w][3] : mxz;
      cnt += sc[w];
    }
    if (cnt) {
      atomicMin(out + 0, mnx); atomicMax(out + 1, mxx);
      atomicMin(out + 2, mnz); atomicMax(out + 3, mxz);
      atomicAdd(reinterpret_cast<unsigned long long*>(out + 4), cnt);
    }
  }
}

// Fresh canvases: topdown = fill (utils.py:472-473), height = -inf (maps.py:2268), mask = false, over cells [0, n) of
// one span (a whole batch of canvases, or one plane of it) by thread `tid` of `nth`.
// Consecutive lanes store consecutive 16-byte words (a thread owning 64 contiguous bytes made every warp
// store touch 32 different lines: 45 % of DRAM peak in ncu).  vec_ok: the three arrays' bases are 16-byte aligned, so
// a cell whose mask byte is 16-byte aligned is aligned in the float arrays too; the head up to the mask's first such
// cell (a plane of h * w cells starts anywhere), the tail, and spans without vec_ok take the scalar loop.
__device__ __forceinline__ void fill_span(float* __restrict__ topdown, float* __restrict__ height,
                                          uint8_t* __restrict__ mask, long long n, float fill, int vec_ok,
                                          long long tid, long long nth) {
  long long head = vec_ok ? (long long)((16 - (reinterpret_cast<uintptr_t>(mask) & 15)) & 15) : n;
  if (head > n) head = n;
  const long long n16 = (n - head) / 16;
  float* t = topdown + head;
  float* h = height ? height + head : nullptr;
  uint8_t* m = mask + head;
  const float4 f4 = make_float4(fill, fill, fill, fill);
  const float4 h4 = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  for (long long i = tid; i < n16 * 4; i += nth) st_stream_f4(t + i * 4, f4);
  if (h)
    for (long long i = tid; i < n16 * 4; i += nth) st_stream_f4(h + i * 4, h4);
  for (long long i = tid; i < n16; i += nth) *reinterpret_cast<uint4*>(m + i * 16) = make_uint4(0u, 0u, 0u, 0u);
  auto one = [&](long long i) {
    topdown[i] = fill;
    if (height) height[i] = -INFINITY;
    mask[i] = 0;
  };
  for (long long i = tid; i < head; i += nth) one(i);
  for (long long i = head + n16 * 16 + tid; i < n; i += nth) one(i);
}

__global__ void __launch_bounds__(kFuseThreads)
fuse_fill_kernel(float* __restrict__ topdown, float* __restrict__ height, uint8_t* __restrict__ mask, long long n,
                 float fill, int vec_ok) {
  fill_span(topdown, height, mask, n, fill, vec_ok, (long long)blockIdx.x * kFuseThreads + threadIdx.x,
            (long long)gridDim.x * kFuseThreads);
}

// MapBuilder.reset_envs: every plane of a sample with done[sample] set gets what fuse_fill_kernel writes, whole (the
// height planes of a value map hold heights at cells whose mask is 0, so the tracked rectangle is not enough); a block
// of another sample's plane leaves at once.  grid = (blocks per plane, planes folded into y).
__global__ void __launch_bounds__(kFuseThreads)
fuse_clear_kernel(float* __restrict__ topdown, float* __restrict__ height, uint8_t* __restrict__ mask,
                  const uint8_t* __restrict__ done, int planes, int C, long long M, float fill, int vec_ok) {
  for (int plane = blockIdx.y; plane < planes; plane += gridDim.y) {
    if (!__ldg(done + plane / C)) continue;
    const long long o = (long long)plane * M;
    fill_span(topdown + o, height ? height + o : nullptr, mask + o, M, fill, vec_ok,
              (long long)blockIdx.x * kFuseThreads + threadIdx.x, (long long)gridDim.x * kFuseThreads);
  }
}

// Block-wide min / max of four per-thread extremes (min, max, min, max); the result is valid in thread 0.
__device__ __forceinline__ void block_reduce_box(float& amin, float& amax, float& bmin, float& bmax) {
  __shared__ float red[kScanThreads / 32][4];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    amin = fminf(amin, __shfl_xor_sync(0xffffffffu, amin, o)); amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    bmin = fminf(bmin, __shfl_xor_sync(0xffffffffu, bmin, o)); bmax = fmaxf(bmax, __shfl_xor_sync(0xffffffffu, bmax, o));
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();  // the previous use of `red` has been read
  if (lane == 0) { red[warp][0] = amin; red[warp][1] = amax; red[warp][2] = bmin; red[warp][3] = bmax; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kScanThreads / 32; ++w) {
      amin = fminf(amin, red[w][0]); amax = fmaxf(amax, red[w][1]);
      bmin = fminf(bmin, red[w][2]); bmax = fmaxf(bmax, red[w][3]);
    }
  }
}

// World map -> new world map (round 2).  A map in the global frame merged into a target in the global frame moves
// every cell by the same whole number of columns and rows — give or take float rounding, which is why the reference's
// per-cell arithmetic is what defines the result.  But that arithmetic is SEPARABLE without transform steps: the
// target column is a function of the source column alone, the target row of the source row alone.  A block evaluates
// both functions — the very float operations of source_point() and quantize_f() — over the plane's rectangle of valid
// cells (a few hundred columns and rows) and accepts the plane when every column moved by one dx and every row by one
// dz and all of them stay inside the canvas.  Then the rectangle is copied densely: whole rows of plain coalesced
// stores (value where the cell is valid and beats the fill, the fill elsewhere) instead of one read-modify-write per
// valid cell into lines of a 0.7 GB canvas the fill kernel has just pushed out of L2.  Only for the first source of a
// call that filled the canvas itself (nothing else has written it yet); anything else takes the per-cell path.
__device__ __forceinline__ bool plane_shift(const DmFuseSource& src, const PlaneCtx& ctx, const DmFuseTarget& tgt, int r0,
                                            int r1, int c0, int c1, int* dx_out, int* dz_out) {
  bool ok = ctx.step0.kind == DM_STEP_NONE && ctx.step1.kind == DM_STEP_NONE && r0 <= r1 && c0 <= c1;
  auto col_of = [&](int c) {  // the x half of source_point + quantize_f
    const float x = __fmul_rn(__fsub_rn((float)c, ctx.woff), src.map_res);
    float xf, zf;
    quantize_f(x, 0.0f, tgt.width_offset, tgt.height_offset, tgt.map_res, tgt.Mh, tgt.flip_h, &xf, &zf);
    return xf;
  };
  auto row_of = [&](int r) {  // the z half
    float zb = (float)r;
    if (src.flip_h) zb = __fsub_rn((float)(src.h - 1), zb);
    const float z = __fmul_rn(__fsub_rn(zb, ctx.hoff), src.map_res);
    float xf, zf;
    quantize_f(0.0f, z, tgt.width_offset, tgt.height_offset, tgt.map_res, tgt.Mh, tgt.flip_h, &xf, &zf);
    return zf;
  };
  int dx = 0, dz = 0;
  if (ok) {
    const float x0 = col_of(c0), z0 = row_of(r0);
    ok = x0 >= 0.0f && x0 < (float)tgt.Mw && z0 >= 0.0f && z0 < (float)tgt.Mh;
    if (ok) {
      dx = (int)x0 - c0;
      dz = (int)z0 - r0;
      for (int c = c0 + threadIdx.x; c <= c1 && ok; c += kScanThreads) {
        const float xf = col_of(c);
        ok = xf >= 0.0f && xf < (float)tgt.Mw && (int)xf - c == dx;
      }
      for (int r = r0 + threadIdx.x; r <= r1 && ok; r += kScanThreads) {
        const float zf = row_of(r);
        ok = zf >= 0.0f && zf < (float)tgt.Mh && (int)zf - r == dz;
      }
    }
  }
  *dx_out = dx;
  *dz_out = dz;
  return __syncthreads_and(ok) != 0;
}

// min_x, max_x, min_z, max_z that pass 1 (fuse_bbox_kernel: source_point + quantize_f with zero offsets) finds for a
// global-frame map in `tgt`'s frame whose valid cells span columns cmin..cmax and rows rmin..rmax (whole numbers held
// in floats).  Every float step is weakly monotone in the column and in the (flipped) row, so the extreme cells give
// the extremes.  Shared by the scatter pass, which tracks the box of the map it writes, and the box rebuild of
// dm_fuse_clear_envs_f32: the same float operations by construction.
__device__ __forceinline__ void tracked_box(const DmFuseTarget& tgt, float cmin, float cmax, float rmin, float rmax,
                                            long long* q) {
  // rows: the dequantised z falls with the row when the map is flipped (maps.py:1081-1083)
  const float zlo = tgt.flip_h ? __fsub_rn((float)(tgt.Mh - 1), rmax) : rmin;
  const float zhi = tgt.flip_h ? __fsub_rn((float)(tgt.Mh - 1), rmin) : rmax;
  auto deq = [&](float bin, float off) { return __fmul_rn(__fsub_rn(bin, off), tgt.map_res); };
  float qx0, qx1, qz0, qz1;
  quantize_f(deq(cmin, tgt.width_offset), deq(zlo, tgt.height_offset), 0.0f, 0.0f, tgt.map_res, 0, 0, &qx0, &qz0);
  quantize_f(deq(cmax, tgt.width_offset), deq(zhi, tgt.height_offset), 0.0f, 0.0f, tgt.map_res, 0, 0, &qx1, &qz1);
  q[0] = f2i64(qx0); q[1] = f2i64(qx1);
  q[2] = f2i64(qz0); q[3] = f2i64(qz1);
}

__global__ void fuse_plane_box_init(int* box, int planes) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < planes; i += gridDim.x * blockDim.x) {
    box[4 * i + 0] = 0x7fffffff; box[4 * i + 1] = -1;  // rows:    min, max
    box[4 * i + 2] = 0x7fffffff; box[4 * i + 3] = -1;  // columns: min, max
  }
}

// mask_inline: the mask (utils.py:489-491: the cell differs from what the canvas was filled with) is
// stored right where a value beats `fill`; with a NaN fill the generic pass below is used instead.
// next_plane_box (optional, (planes, 4) int32 = row min / max, column min / max, initialised by fuse_plane_box_init):
// the rectangle of every plane of the map written here that holds its valid cells — what a later merge needs to scan
// when this map is one of its sources (DmFuseSource.plane_box).
__global__ void __launch_bounds__(kScanThreads, 1024 / kScanThreads)
fuse_scatter_kernel(const __grid_constant__ DmFuseSource src, int planes, int C, const DmFuseTarget tgt,
                    float* __restrict__ topdown, float* __restrict__ height, uint8_t* __restrict__ mask,
                    int mask_inline, long long* __restrict__ next_bbox, int* __restrict__ next_plane_box,
                    int fresh_canvas) {
  __shared__ PlaneCtx ctx;
  // next_bbox: what pass 1 of a FOLLOWING merge would find for the map written here, taken as a global-frame
  // source of the same resolution: min / max over its valid cells of quantize0(dequantize(cell)) (maps.py:1081-1086,
  // 2159-2165) — a function of the cell and this target's offsets only, and non-decreasing in the column and in the
  // (flipped) row: every float step (int → float, − offset, × res, / res, + 0.5, floor) is weakly monotone.  So the
  // extreme columns / rows that were marked valid are all that is tracked per cell (whole numbers held in floats);
  // the four bins are evaluated once per block.
  float cmin = INFINITY, cmax = -INFINITY, rmin = INFINITY, rmax = -INFINITY;
  const long long M = (long long)tgt.Mh * tgt.Mw;
  const int n = src.h * src.w;
  int loaded = -1;
  for (int plane = blockIdx.y; plane < planes; plane += gridDim.y) {
    const int smp = plane / C, ch = plane - smp * C;
    if (smp != loaded) { load_plane_ctx(src, smp, &ctx); loaded = smp; }
    const float* hplane = src.height + (long long)smp * src.height_bstride + (long long)ch * src.height_cstride;
    const float* vplane = src.values ? src.values + (long long)plane * n : nullptr;
    float* tplane = topdown + (long long)plane * M;
    float* oplane = height ? height + (long long)plane * M : nullptr;
    uint8_t* mplane = mask + (long long)plane * M;
    float pcmin = INFINITY, pcmax = -INFINITY, prmin = INFINITY, prmax = -INFINITY;  // this plane's marked cells
    bool dense = false;
    if (fresh_canvas && mask_inline && src.plane_box) {  // block-uniform
      const int4 bx = __ldg(reinterpret_cast<const int4*>(src.plane_box) + plane);  // rmin, rmax, cmin, cmax
      const int r0 = max(bx.x, 0), r1 = min(bx.y, src.h - 1), c0 = max(bx.z, 0), c1 = min(bx.w, src.w - 1);
      int dx, dz;
      dense = plane_shift(src, ctx, tgt, r0, r1, c0, c1, &dx, &dz);
      if (dense) {
        const uint8_t* smask = src.mask + (long long)plane * n;
        const int wbox = c1 - c0 + 1;
        // a block takes whole rows of the rectangle; a thread four cells of the row per round (their loads in flight
        // together), consecutive lanes consecutive cells
        for (int r = r0 + blockIdx.x; r <= r1; r += gridDim.x) {
          const int srow = r * src.w + c0, trow = (r + dz) * tgt.Mw + (c0 + dx);
          for (int cb = threadIdx.x; cb < wbox; cb += 4 * kScanThreads) {
            uint8_t m[4];
            float y[4], v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int ci = cb + k * kScanThreads;
              m[k] = ci < wbox ? smask[srow + ci] : (uint8_t)0;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int ci = cb + k * kScanThreads;
              y[k] = m[k] ? hplane[srow + ci] : 0.0f;
              v[k] = (m[k] && vplane) ? vplane[srow + ci] : y[k];  // maps.py:2214-2216
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int ci = cb + k * kScanThreads;
              if (ci >= wbox) continue;
              float out = tgt.fill_value, hout = -INFINITY;
              uint8_t mk = 0;
              if (m[k]) {
                if (v[k] == v[k] && better(v[k], tgt.fill_value, tgt.reduction)) {  // what the atomic leaves in a cell that held fill
                  out = v[k];
                  mk = 1;
                  const float xf = (float)(c0 + ci + dx), zf = (float)(r + dz);
                  pcmin = fminf(pcmin, xf); pcmax = fmaxf(pcmax, xf);
                  prmin = fminf(prmin, zf); prmax = fmaxf(prmax, zf);
                }
                if (y[k] == y[k]) hout = fmaxf(hout, y[k]);  // maps.py:2258-2271: max against -inf
              }
              tplane[trow + ci] = out;
              mplane[trow + ci] = mk;
              if (oplane) oplane[trow + ci] = hout;
            }
          }
        }
      }
    }
    if (!dense) for_valid_cells(src, plane, [&](int cell, int r, int c) {
      const V3 p = source_point(src, ctx, hplane, cell, r, c);
      float xf, zf;  // maps.py:2232-2238
      quantize_f(p.x, p.z, tgt.width_offset, tgt.height_offset, tgt.map_res, tgt.Mh, tgt.flip_h, &xf, &zf);
      if (!(xf >= 0.0f && xf < (float)tgt.Mw && zf >= 0.0f && zf < (float)tgt.Mh)) return;
      const int o = (int)zf * tgt.Mw + (int)xf;
      const float v = vplane ? vplane[cell] : p.y;  // maps.py:2214-2216
      if (v == v) {
        if (tgt.reduction) atomic_min_f32(tplane + o, v); else atomic_max_f32(tplane + o, v);
        if (mask_inline && better(v, tgt.fill_value, tgt.reduction)) {
          mplane[o] = 1;
          pcmin = fminf(pcmin, xf); pcmax = fmaxf(pcmax, xf);
          prmin = fminf(prmin, zf); prmax = fmaxf(prmax, zf);
        }
      }
      if (oplane && p.y == p.y) atomic_max_f32(oplane + o, p.y);  // maps.py:2258-2271
    });
    cmin = fminf(cmin, pcmin); cmax = fmaxf(cmax, pcmax);
    rmin = fminf(rmin, prmin); rmax = fmaxf(rmax, prmax);
    if (next_plane_box) {  // block-uniform branch: one set of atomics per block and plane it marked a cell in
      block_reduce_box(prmin, prmax, pcmin, pcmax);
      if (threadIdx.x == 0 && pcmin <= pcmax) {
        atomicMin(next_plane_box + 4 * plane + 0, (int)prmin); atomicMax(next_plane_box + 4 * plane + 1, (int)prmax);
        atomicMin(next_plane_box + 4 * plane + 2, (int)pcmin); atomicMax(next_plane_box + 4 * plane + 3, (int)pcmax);
      }
    }
  }
  if (next_bbox) {  // warp, then block reduction; one set of atomics per block that marked a cell
    block_reduce_box(cmin, cmax, rmin, rmax);
    if (threadIdx.x == 0) {
      if (cmin <= cmax) {
        long long q[4];
        tracked_box(tgt, cmin, cmax, rmin, rmax, q);
        atomicMin(next_bbox + 0, q[0]); atomicMax(next_bbox + 1, q[1]);
        atomicMin(next_bbox + 2, q[2]); atomicMax(next_bbox + 3, q[3]);
        atomicAdd(reinterpret_cast<unsigned long long*>(next_bbox + 4), 1ull);
      }
    }
  }
}

// dm_fuse_clear_envs_f32's rectangles and box, one block: the rectangles of the cleared planes become empty
// (fuse_plane_box_init's sentinel), the others stay, and `box` (may be NULL) becomes what the scatter pass would have
// left for a map holding only the surviving planes: tracked_box() of their extremes, counting the non-empty planes
// (zero iff no valid cell is left).  With nothing cleared it stays as it is.
__global__ void __launch_bounds__(kScanThreads)
fuse_clear_boxes_kernel(const uint8_t* __restrict__ done, int planes, int C, const DmFuseTarget tgt,
                        int* __restrict__ plane_box, long long* __restrict__ box) {
  __shared__ unsigned int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  float cmin = INFINITY, cmax = -INFINITY, rmin = INFINITY, rmax = -INFINITY;
  unsigned int cnt = 0;
  int cleared = 0;
  for (int p = threadIdx.x; p < planes; p += kScanThreads) {
    int4* pb = reinterpret_cast<int4*>(plane_box) + p;  // rmin, rmax, cmin, cmax
    if (__ldg(done + p / C)) {
      *pb = make_int4(0x7fffffff, -1, 0x7fffffff, -1);
      cleared = 1;
      continue;
    }
    const int4 bx = *pb;
    if (bx.y < bx.x || bx.w < bx.z) continue;  // no valid cell
    rmin = fminf(rmin, (float)bx.x); rmax = fmaxf(rmax, (float)bx.y);
    cmin = fminf(cmin, (float)bx.z); cmax = fmaxf(cmax, (float)bx.w);
    ++cnt;
  }
  if (!box) return;  // block-uniform
  if (!__syncthreads_or(cleared)) return;  // nothing cleared: the box stays as the scatter pass left it, count included
  if (cnt) atomicAdd(&s_cnt, cnt);
  block_reduce_box(cmin, cmax, rmin, rmax);  // its barriers order the count's atomics before thread 0 reads it
  if (threadIdx.x == 0) {
    if (s_cnt) {
      long long q[4];
      tracked_box(tgt, cmin, cmax, rmin, rmax, q);
      for (int i = 0; i < 4; ++i) box[i] = q[i];
      box[4] = s_cnt;
    } else {  // what fuse_bbox_init starts from
      box[0] = 0x7fffffffffffffffLL; box[1] = (long long)0x8000000000000000ULL;
      box[2] = 0x7fffffffffffffffLL; box[3] = (long long)0x8000000000000000ULL;
      box[4] = 0;
    }
  }
}

static dim3 plane_grid(const DmFuseSource& s, int planes);

// sum / mean / prod (utils.py:70-76): the merged value of a cell depends on the order of its hits, which is the
// order of the reference's concatenated point cloud (_merge_point_clouds, maps.py:2071-2127: per (sample, channel)
// row the cells of source 0 in row-major order, then those of source 1, ...).  Every point gets the key of its target
// cell at position plane * points_per_plane + source offset + cell, and dm_ordered.cu folds each cell's hits in
// ascending position.  The height map of a value-map merge stays an (order-independent) atomic max.
__global__ void __launch_bounds__(kScanThreads)
fuse_keys_kernel(const __grid_constant__ DmFuseSource src, int planes, int C, const DmFuseTarget tgt, long long off,
                 long long points_per_plane, unsigned long long* __restrict__ keys, float* __restrict__ vals,
                 float* __restrict__ height) {
  __shared__ PlaneCtx ctx;
  const long long M = (long long)tgt.Mh * tgt.Mw;
  const int n = src.h * src.w;
  int loaded = -1;
  for (int plane = blockIdx.y; plane < planes; plane += gridDim.y) {
    const int smp = plane / C, ch = plane - smp * C;
    if (smp != loaded) { load_plane_ctx(src, smp, &ctx); loaded = smp; }
    const float* hplane = src.height + (long long)smp * src.height_bstride + (long long)ch * src.height_cstride;
    const float* vplane = src.values ? src.values + (long long)plane * n : nullptr;
    const uint8_t* mplane = src.mask + (long long)plane * n;
    for (int cell = blockIdx.x * kScanThreads + threadIdx.x; cell < n; cell += gridDim.x * kScanThreads) {
      const long long pos = (long long)plane * points_per_plane + off + cell;
      unsigned long long key = ~0ull;
      float v = 0.0f;
      if (mplane[cell]) {
        const int r = cell / src.w;
        const V3 p = source_point(src, ctx, hplane, cell, r, cell - r * src.w);
        float xf, zf;  // maps.py:2232-2238
        quantize_f(p.x, p.z, tgt.width_offset, tgt.height_offset, tgt.map_res, tgt.Mh, tgt.flip_h, &xf, &zf);
        if (xf >= 0.0f && xf < (float)tgt.Mw && zf >= 0.0f && zf < (float)tgt.Mh) {
          const long long o = (long long)plane * M + (long long)zf * tgt.Mw + (long long)xf;
          key = (unsigned long long)o;
          v = vplane ? vplane[cell] : p.y;  // maps.py:2214-2216
          if (height && p.y == p.y) atomic_max_f32(height + o, p.y);  // maps.py:2258-2271
        }
      }
      keys[pos] = key;
      vals[pos] = v;
    }
  }
}

static int launch_ordered(const DmFuseSource* sources, int n_sources, int b, int C, const DmFuseTarget& tgt,
                          float* topdown, uint8_t* mask, float* height, cudaStream_t stream) {
  const long long planes = (long long)b * C, M = (long long)tgt.Mh * tgt.Mw;
  long long per_plane = 0;
  for (int i = 0; i < n_sources; ++i) per_plane += (long long)sources[i].h * sources[i].w;
  const long long total = planes * per_plane;
  if (total >= (1ll << 31)) return DM_EINVAL;
  if (total == 0) return DM_OK;
  unsigned long long* keys = nullptr;
  float* vals = nullptr;
  DM_CUDA_OK(cudaMallocAsync(&keys, (size_t)total * 8, stream));
  DM_CUDA_OK(cudaMallocAsync(&vals, (size_t)total * 4, stream));
  long long off = 0;
  for (int i = 0; i < n_sources; ++i) {
    fuse_keys_kernel<<<plane_grid(sources[i], (int)planes), kScanThreads, 0, stream>>>(sources[i], (int)planes, C, tgt, off,
                                                                                        per_plane, keys, vals, height);
    DM_LAUNCHED();
    off += (long long)sources[i].h * sources[i].w;
  }
  const int rc = ordered_reduce(keys, vals, total, bits_for((unsigned long long)(planes * M)), tgt.reduction, topdown,
                                mask, stream);
  DM_CUDA_OK(cudaFreeAsync(keys, stream));
  DM_CUDA_OK(cudaFreeAsync(vals, stream));
  return rc;
}

__global__ void __launch_bounds__(kFuseThreads)
changed_mask_kernel(const float* __restrict__ canvas, long long n, float fill, uint8_t* __restrict__ mask) {
  for (long long i = (long long)blockIdx.x * kFuseThreads + threadIdx.x; i < n;
       i += (long long)gridDim.x * kFuseThreads) {
    float d = fabsf(__fsub_rn(canvas[i], fill));  // utils.py:489-491
    if (d != d) d = 0.0f;
    mask[i] = d != 0.0f;
  }
}

static int check_sources(const DmFuseSource* sources, int n, int b, int C) {
  if (!sources || n <= 0 || n > kMaxSources || b <= 0 || C <= 0) return DM_EINVAL;
  if ((long long)b * C >= (1ll << 31)) return DM_EINVAL;
  for (int i = 0; i < n; ++i) {
    const DmFuseSource& s = sources[i];
    if (!s.height || !s.mask || !s.width_offset || !s.height_offset || !s.steps || s.h <= 0 || s.w <= 0)
      return DM_EINVAL;
    if ((long long)s.h * s.w >= (1ll << 30)) return DM_EINVAL;
  }
  return DM_OK;
}

// (blocks per plane, planes folded into y): about `waves` waves of 8 resident 256-thread CTAs per SM in total
static dim3 plane_grid(const DmFuseSource& s, int planes) {
  constexpr int waves = 2, max_gy = 65535;
  const long long groups = ((long long)s.h * s.w + 2 * kGroup - 1) / kGroup;
  const int gy = planes < max_gy ? planes : max_gy;
  long long gx = (((long long)sm_count() * 8 * waves + gy - 1) / gy) * (256 / kScanThreads);
  long long gx_max = (groups + kScanThreads - 1) / kScanThreads;
  // ... and a block should have a few thousand cells to scan: its fixed costs (context load, box reductions, their
  // barriers and atomics) are ~10 us, which for a 400 x 400 local map split 148 ways was most of the kernel
  const long long by_work = ((long long)s.h * s.w + kMinCellsPerBlock - 1) / kMinCellsPerBlock;
  if (gx_max > by_work) gx_max = by_work;
  if (gx > gx_max) gx = gx_max;
  if (gx < 1) gx = 1;
  return dim3((unsigned)gx, (unsigned)gy);
}

static unsigned grid_for(long long items) {
  long long blocks = (items + kFuseThreads - 1) / kFuseThreads;
  const long long cap = (long long)sm_count() * 8 * 4;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

// fresh: the canvases hold nothing but what fuse_fill_kernel wrote (the caller filled them itself): the first source
// may then write its cells with plain stores (plane_shift).
static int launch_scatter(const DmFuseSource* sources, int n_sources, int b, int C, const DmFuseTarget& tgt,
                          float* topdown, uint8_t* mask, float* height, int mask_inline, cudaStream_t stream,
                          long long* next_bbox = nullptr, int* next_plane_box = nullptr, int fresh = 0) {
  for (int i = 0; i < n_sources; ++i) {
    const int dense = (fresh && i == 0 && g_dense_shift) ? 1 : 0;
    dim3 grid = plane_grid(sources[i], b * C);
    // the dense copy moves a few hundred rows per plane: with ~150 blocks per plane a block copies 3 rows and spends
    // its life in per-block fixed costs (context load, shift test, two box reductions: 4 waves of ~10 us); one wave of
    // fatter blocks instead
    if (dense && mask_inline && sources[i].plane_box) {
      const unsigned per_plane = (unsigned)((sm_count() * 8 + grid.y - 1) / grid.y);
      if (grid.x > per_plane) grid.x = per_plane > 0 ? per_plane : 1;
    }
    fuse_scatter_kernel<<<grid, kScanThreads, 0, stream>>>(
        sources[i], b * C, C, tgt, topdown, height, mask, mask_inline, next_bbox, next_plane_box, dense);
    DM_LAUNCHED();
  }
  return DM_OK;
}

}  // namespace dm

using namespace dm;

extern "C" void dm_debug_set_dense_shift(int32_t on) { dm::g_dense_shift = on ? 1 : 0; }

int dm::fuse_bbox_accumulate(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C, float target_res,
                             int64_t* bbox, cudaStream_t stream) {
  if (!bbox) return DM_EINVAL;
  const int rc = check_sources(sources, n_sources, b, C);
  if (rc != DM_OK) return rc;
  for (int i = 0; i < n_sources; ++i) {
    fuse_bbox_kernel<<<plane_grid(sources[i], b * C), kScanThreads, 0, stream>>>(sources[i], b * C, C, target_res,
                                                                               reinterpret_cast<long long*>(bbox));
    DM_LAUNCHED();
  }
  return DM_OK;
}

int dm::hmap_resolve_with_bbox(uint32_t* planes, unsigned long long slot_words, const DmProjCfg* cfg, int32_t b,
                               float* topdown, uint8_t* mask, const DmFuseSource* local, float target_res,
                               const int64_t* seed, int64_t* bbox, cudaStream_t stream) {
  if (!planes || !cfg || !topdown || !mask || !local || !bbox || b <= 0) return DM_EINVAL;
  const int rc = check_sources(local, 1, b, 1);
  if (rc != DM_OK) return rc;
  if (local->h != cfg->Mh || local->w != cfg->Mw) return DM_EINVAL;
  fuse_bbox_init<<<1, 1, 0, stream>>>(reinterpret_cast<long long*>(bbox), reinterpret_cast<const long long*>(seed));
  DM_LAUNCHED();
  const int M = cfg->Mh * cfg->Mw;
  const int vec = (M % 4 == 0) && reinterpret_cast<uintptr_t>(topdown) % 16 == 0 && reinterpret_cast<uintptr_t>(mask) % 4 == 0;
  // blocks of 4 x 1024 cells: few enough that their five same-address atomics stay cheap
  const unsigned gx = (unsigned)((M + 4095) / 4096);
  hmap_resolve_bbox_kernel<<<dim3(gx > 0 ? gx : 1, b), 256, 0, stream>>>(planes, slot_words, *cfg, vec, topdown, mask,
                                                                         *local, target_res,
                                                                         reinterpret_cast<long long*>(bbox));
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_fuse_bbox_i64(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                                float target_res, int64_t* out, void* stream_) {
  DM_TRACE();
  return dm_fuse_bbox_seeded_i64(sources, n_sources, b, C, target_res, nullptr, out, stream_);
}

extern "C" int dm_fuse_bbox_seeded_i64(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                                       float target_res, const int64_t* seed, int64_t* out, void* stream_) {
  DM_TRACE();
  if (!out) return DM_EINVAL;
  if (n_sources == 0 && !seed) return DM_EINVAL;
  if (n_sources != 0) {
    const int rc = check_sources(sources, n_sources, b, C);
    if (rc != DM_OK) return rc;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  fuse_bbox_init<<<1, 1, 0, stream>>>(reinterpret_cast<long long*>(out), reinterpret_cast<const long long*>(seed));
  DM_LAUNCHED();
  for (int i = 0; i < n_sources; ++i) {
    // (fewer, longer blocks that walk several planes each were tried for the five same-address atomics at the end of
    // every block: slower, 103-113 us instead of 76 us for the config-4 world map — the planes are unevenly filled)
    fuse_bbox_kernel<<<plane_grid(sources[i], b * C), kScanThreads, 0, stream>>>(sources[i], b * C, C, target_res,
                                                                               reinterpret_cast<long long*>(out));
    DM_LAUNCHED();
  }
  return DM_OK;
}

extern "C" int dm_fuse_scatter_f32(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                                   const DmFuseTarget* target, float* topdown, uint8_t* mask, float* height,
                                   void* stream_) {
  DM_TRACE();
  return dm_fuse_scatter_track_f32(sources, n_sources, b, C, target, topdown, mask, height, nullptr, nullptr, stream_);
}

extern "C" int dm_fuse_scatter_track_f32(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                                         const DmFuseTarget* target, float* topdown, uint8_t* mask, float* height,
                                         int64_t* next_bbox, int32_t* next_plane_box, void* stream_) {
  DM_TRACE();
  return fuse_scatter_track(sources, n_sources, b, C, target, topdown, mask, height, next_bbox, next_plane_box, 0,
                            stream_);
}

// prefilled: the canvases already hold what fuse_fill_kernel writes (dm_builder_plot_prefill queued it) — untouched since
int dm::fuse_scatter_track(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                           const DmFuseTarget* target, float* topdown, uint8_t* mask, float* height,
                           int64_t* next_bbox, int32_t* next_plane_box, int prefilled, void* stream_) {
  if (!target || !topdown || !mask || target->Mh <= 0 || target->Mw <= 0) return DM_EINVAL;
  if (target->reduction < 0 || target->reduction > 4) return DM_EINVAL;
  if (target->reduction >= 2 && (next_bbox || next_plane_box)) return DM_EINVAL;  // tracking assumes "mask = beats fill"
  const int rc = check_sources(sources, n_sources, b, C);
  if (rc != DM_OK) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long n_out = (long long)b * C * target->Mh * target->Mw;
  if ((long long)target->Mh * target->Mw >= (1ll << 31)) return DM_EINVAL;
  const int vec_ok = reinterpret_cast<uintptr_t>(topdown) % 16 == 0 && reinterpret_cast<uintptr_t>(mask) % 16 == 0 &&
                     (!height || reinterpret_cast<uintptr_t>(height) % 16 == 0);
  const int mask_inline = target->fill_value == target->fill_value;  // not NaN
  if (!prefilled) {
    fuse_fill_kernel<<<grid_for((n_out + 3) / 4), kFuseThreads, 0, stream>>>(topdown, height, mask, n_out,
                                                                             target->fill_value, vec_ok);
    DM_LAUNCHED();
  }
  if (target->reduction >= 2)  // order-dependent reductions: the reference's point order, bit for bit
    return launch_ordered(sources, n_sources, b, C, *target, topdown, mask, height, stream);
  if (next_bbox || next_plane_box) {
    if (!mask_inline) return DM_EINVAL;  // NaN fill: the mask comes from the compare pass, nothing to track
    if (next_bbox) {
      fuse_bbox_init<<<1, 1, 0, stream>>>(reinterpret_cast<long long*>(next_bbox));
      DM_LAUNCHED();
    }
    if (next_plane_box) {
      fuse_plane_box_init<<<(b * C + 255) / 256, 256, 0, stream>>>(next_plane_box, b * C);
      DM_LAUNCHED();
    }
  }
  const int rs = launch_scatter(sources, n_sources, b, C, *target, topdown, mask, height, mask_inline, stream,
                                reinterpret_cast<long long*>(next_bbox), next_plane_box, 1);
  if (rs != DM_OK) return rs;
  if (!mask_inline) {
    changed_mask_kernel<<<grid_for(n_out), kFuseThreads, 0, stream>>>(topdown, n_out, target->fill_value, mask);
    DM_LAUNCHED();
  }
  return DM_OK;
}

// Opt-in fixed-canvas merge (no reference equivalent of the call; the semantics are those of the
// reference's project(..., canvas=, canvas_masks=), maps.py:1089-1173 / utils.py:462-491): the valid
// cells of the sources are max-merged IN PLACE into canvases that already hold a world map.  No
// bounding box, no host sync, no reallocation: one launch.  Invariant kept: mask == (cell != fill).
extern "C" int dm_fuse_inplace_f32(const DmFuseSource* sources, int32_t n_sources, int32_t b, int32_t C,
                                   const DmFuseTarget* target, float* topdown, uint8_t* mask, float* height,
                                   void* stream_) {
  DM_TRACE();
  if (!target || !topdown || !mask || target->Mh <= 0 || target->Mw <= 0) return DM_EINVAL;
  if (target->reduction < 0 || target->reduction > 4) return DM_EINVAL;
  if (!(target->fill_value == target->fill_value)) return DM_EINVAL;  // NaN fill has no in-place mask rule
  const int rc = check_sources(sources, n_sources, b, C);
  if (rc != DM_OK) return rc;
  if ((long long)target->Mh * target->Mw >= (1ll << 31)) return DM_EINVAL;
  if (target->reduction >= 2)  // sum / mean / prod into the existing canvases: mask |= "cell changed" (utils.py:489-491)
    return launch_ordered(sources, n_sources, b, C, *target, topdown, mask, height, static_cast<cudaStream_t>(stream_));
  return launch_scatter(sources, n_sources, b, C, *target, topdown, mask, height, 1, static_cast<cudaStream_t>(stream_));
}

/* Fills fresh world canvases for dm_fuse_inplace_f32: topdown = fill_value, height = -inf (may be NULL), mask = 0. */
extern "C" int dm_fuse_canvas_init_f32(float* topdown, uint8_t* mask, float* height, int64_t n, float fill_value,
                                       void* stream_) {
  DM_TRACE();
  if (!topdown || !mask || n < 0) return DM_EINVAL;
  if (n == 0) return DM_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int vec_ok = reinterpret_cast<uintptr_t>(topdown) % 16 == 0 && reinterpret_cast<uintptr_t>(mask) % 16 == 0 &&
                     (!height || reinterpret_cast<uintptr_t>(height) % 16 == 0);
  fuse_fill_kernel<<<grid_for((n + 3) / 4), kFuseThreads, 0, stream>>>(topdown, height, mask, n, fill_value, vec_ok);
  DM_LAUNCHED();
  return DM_OK;
}

/* MapBuilder.reset_envs: the planes of the samples with done[s] set become fresh canvas, their tracked rectangles empty,
 * and the tracked box is rebuilt from the surviving rectangles.  `done` is read on the device only. */
extern "C" int dm_fuse_clear_envs_f32(float* topdown, float* height, uint8_t* mask, int32_t b, int32_t C,
                                      const uint8_t* done, const DmFuseTarget* map, int32_t* plane_box, int64_t* box,
                                      void* stream_) {
  DM_TRACE();
  if (!topdown || !mask || !done || !map || b <= 0 || C <= 0 || map->Mh <= 0 || map->Mw <= 0) return DM_EINVAL;
  if ((long long)b * C >= (1ll << 31) || (long long)map->Mh * map->Mw >= (1ll << 31)) return DM_EINVAL;
  if (map->reduction < 0 || map->reduction > 4) return DM_EINVAL;
  if (box && !plane_box) return DM_EINVAL;  // the box is rebuilt from the rectangles
  // tracking assumes "mask = beats fill"
  if ((box || plane_box) && (!(map->fill_value == map->fill_value) || map->reduction >= 2)) return DM_EINVAL;
  if (reinterpret_cast<uintptr_t>(plane_box) % 16 != 0) return DM_EINVAL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int planes = b * C;
  const long long M = (long long)map->Mh * map->Mw;
  const int vec_ok = reinterpret_cast<uintptr_t>(topdown) % 16 == 0 && reinterpret_cast<uintptr_t>(mask) % 16 == 0 &&
                     (!height || reinterpret_cast<uintptr_t>(height) % 16 == 0);
  // a block stores 1024 cells per round: a few rounds per block, and at most two blocks per SM for one plane (the
  // blocks of planes that are not cleared cost a launch slot each)
  long long gx = (M + 4095) / 4096;
  if (gx > 2ll * sm_count()) gx = 2ll * sm_count();
  const unsigned gy = planes < 65535 ? (unsigned)planes : 65535u;
  fuse_clear_kernel<<<dim3((unsigned)gx, gy), kFuseThreads, 0, stream>>>(topdown, height, mask, done, planes, C, M,
                                                                         map->fill_value, vec_ok);
  DM_LAUNCHED();
  if (plane_box) {
    fuse_clear_boxes_kernel<<<1, kScanThreads, 0, stream>>>(done, planes, C, *map, plane_box,
                                                            reinterpret_cast<long long*>(box));
    DM_LAUNCHED();
  }
  return DM_OK;
}
