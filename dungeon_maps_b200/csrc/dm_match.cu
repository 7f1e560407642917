// score_poses: per-environment match counts of a local window against the planes of a global-frame map at candidate
// poses (include/dungeon_maps_b200.h: dm_score_poses_i32).  score[i, c, k] counts the True window cells whose cell of
// TopdownMap.select_egocentric at candidate k (map_dequantize with the window offsets -> local_to_global_space ->
// map_quantize with the source offsets) lands inside the source on a True cell of plane c.  The geometry is the crop's
// (dequantize_f, apply_step, quantize_f), so the counted cells are exactly the True cells of crop_egocentric_map.
//
// Two kernels on the caller's stream, no grid sync, no host sync, no atomics:
//   1. match_compact_kernel  one CTA per window plane: the linear indices of its True cells in raster order, and their
//                            count, into stream-ordered scratch.  Only True cells can add to a score.
//   2. match_score_kernel    one CTA per (window plane, group of candidates, group of planes): each thread holds a few
//                            listed cells, applies each candidate's block to them, and tests the plane bytes; the hits
//                            of a warp are summed with one __reduce_add_sync per (candidate, plane) and kept by the
//                            lane that owns that pair, so at most 32 pairs go to a CTA.  One int32 store per pair.
// Counts are integers: the result does not depend on the order of the sums.
#include "dm_common.cuh"

namespace dm {
namespace {

constexpr int kCompactThreads = 256;
constexpr int kCompactPer = 16;                           // cells per thread per tile (one uint4 of shared memory)
constexpr int kCompactTile = kCompactThreads * kCompactPer;
constexpr int kScoreThreads = 256;
constexpr int kScoreCells = 4;                            // listed cells per thread per tile
constexpr int kScoreTile = kScoreThreads * kScoreCells;
constexpr int kPairs = 32;                                // (candidate, plane) pairs per CTA: one per lane

// Pass 1.  Tiles of 4096 cells: a coalesced copy to shared memory, then each thread takes 16 consecutive cells, counts
// its True ones, and a block scan gives every thread its place in the list.
__global__ void __launch_bounds__(kCompactThreads) match_compact_kernel(const uint8_t* __restrict__ window,
                                                                        long long n_lists, int hw,
                                                                        int* __restrict__ cells,
                                                                        int* __restrict__ counts) {
  __shared__ __align__(16) uint8_t tile[kCompactTile];
  __shared__ int warp_sum[kCompactThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (long long l = blockIdx.x; l < n_lists; l += gridDim.x) {
    const uint8_t* win = window + l * hw;
    int* out = cells + l * hw;
    int total = 0;
    for (long long base = 0; base < hw; base += kCompactTile) {
#pragma unroll
      for (int j = 0; j < kCompactPer; ++j) {
        const long long q = base + j * kCompactThreads + tid;
        tile[j * kCompactThreads + tid] = q < hw ? win[q] : (uint8_t)0;
      }
      __syncthreads();
      const uint4 v = reinterpret_cast<const uint4*>(tile)[tid];
      const unsigned words[4] = {v.x, v.y, v.z, v.w};
      unsigned bits = 0;
#pragma unroll
      for (int j = 0; j < kCompactPer; ++j)
        if ((words[j >> 2] >> (8 * (j & 3))) & 0xffu) bits |= 1u << j;
      const int mine = __popc(bits);
      int incl = mine;                                    // inclusive scan over the warp, then over the warps
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += up;
      }
      if (lane == 31) warp_sum[warp] = incl;
      __syncthreads();
      int before = 0, all = 0;
#pragma unroll
      for (int w = 0; w < kCompactThreads / 32; ++w) {
        const int s = warp_sum[w];
        before += w < warp ? s : 0;
        all += s;
      }
      int pos = total + before + incl - mine;
      const int first = (int)base + kCompactPer * tid;    // < hw whenever a bit is set
      while (bits) {
        const int j = __ffs(bits) - 1;
        bits &= bits - 1;
        out[pos++] = first + j;
      }
      total += all;
      __syncthreads();                                    // tile and warp_sum are rewritten next
    }
    if (tid == 0) counts[l] = total;
  }
}

// Pass 2.  Block index = (list, plane group, candidate group), candidate group fastest so that neighbouring CTAs read
// the same region of the same environment's planes.  A list is window plane p of environment i (n_wp planes per
// environment: 1, shared by all C planes, or C, one per plane).  Pair (g, c) of the CTA is lane g * pw + c.
__global__ void __launch_bounds__(kScoreThreads) match_score_kernel(
    const uint8_t* __restrict__ planes, int C, int Hs, int Ws, float res, int flip_h, int n_wp, int h, int w,
    const float* __restrict__ samples, int n, const int* __restrict__ cells, const int* __restrict__ counts,
    long long n_lists, int plane_groups, int pw, int cand_groups, int* __restrict__ scores) {
  __shared__ __align__(16) float blk[kPairs * DM_EGO_SAMPLE_WORDS];
  __shared__ int warp_acc[kScoreThreads / 32][32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = kPairs / pw;
  const long long plane = (long long)Hs * Ws;
  const long long hw = (long long)h * w;
  const long long n_blocks = n_lists * plane_groups * cand_groups;
  for (long long bid = blockIdx.x; bid < n_blocks; bid += gridDim.x) {
    const int cg = (int)(bid % cand_groups);
    const long long rest = bid / cand_groups;
    const int pg = (int)(rest % plane_groups);
    const long long l = rest / plane_groups;
    const long long i = l / n_wp;
    const int c0 = n_wp == 1 ? pg * pw : (int)(l - i * n_wp);
    const int nc = n_wp == 1 ? min(pw, C - c0) : 1;
    const int k0 = cg * G;
    const int ng = min(G, n - k0);
    const float* src = samples + ((long long)i * n + k0) * DM_EGO_SAMPLE_WORDS;
    for (int q = tid; q < ng * DM_EGO_SAMPLE_WORDS; q += kScoreThreads) blk[q] = src[q];
    __syncthreads();
    const int count = counts[l];
    const int* list = cells + l * hw;
    const uint8_t* pl = planes + ((long long)i * C + c0) * plane;
    int acc = 0;
    for (long long base = 0; base < count; base += kScoreTile) {
      float cf[kScoreCells], rf[kScoreCells];
      bool ok[kScoreCells];
#pragma unroll
      for (int t = 0; t < kScoreCells; ++t) {
        const long long q = base + t * kScoreThreads + tid;
        ok[t] = q < count;
        const int idx = ok[t] ? list[q] : 0;
        const int r = idx / w;
        cf[t] = (float)(idx - r * w);
        rf[t] = (float)r;
      }
      for (int g = 0; g < ng; ++g) {
        const float* b = blk + g * DM_EGO_SAMPLE_WORDS;
        const DmStep& step = *reinterpret_cast<const DmStep*>(b);
        const float src_woff = b[16], src_hoff = b[17], woff = b[18], hoff = b[19];
        int off[kScoreCells];
        bool in[kScoreCells];
#pragma unroll
        for (int t = 0; t < kScoreCells; ++t) {
          float lx, lz, xf, zf;
          dequantize_f(cf[t], rf[t], woff, hoff, res, h, flip_h, &lx, &lz);
          const V3 p = apply_step(step, V3{lx, 0.0f, lz});
          quantize_f(p.x, p.z, src_woff, src_hoff, res, Hs, flip_h, &xf, &zf);
          in[t] = ok[t] && xf >= 0.0f && xf < (float)Ws && zf >= 0.0f && zf < (float)Hs;
          off[t] = in[t] ? (int)zf * Ws + (int)xf : 0;
        }
        for (int c = 0; c < nc; ++c) {
          const uint8_t* pc = pl + c * plane;
          int hits = 0;
#pragma unroll
          for (int t = 0; t < kScoreCells; ++t) hits += (int)(in[t] & (pc[off[t]] != 0));   // off is 0 outside
          hits = __reduce_add_sync(0xffffffffu, hits);
          if (lane == g * pw + c) acc += hits;
        }
      }
    }
    warp_acc[warp][lane] = acc;
    __syncthreads();
    if (tid < 32) {
      int sum = 0;
#pragma unroll
      for (int wp = 0; wp < kScoreThreads / 32; ++wp) sum += warp_acc[wp][tid];
      const int g = tid / pw, c = tid - g * pw;
      if (g < ng && c < nc) scores[((long long)i * C + c0 + c) * n + k0 + g] = sum;
    }
    __syncthreads();                                      // blk and warp_acc are rewritten next
  }
}

}  // namespace
}  // namespace dm

using namespace dm;

extern "C" int dm_score_poses_i32(const uint8_t* planes, int32_t b, int32_t C, int32_t Hs, int32_t Ws, float map_res,
                                  int32_t flip_h, const uint8_t* window, int32_t window_planes, int32_t h, int32_t w,
                                  const float* samples, int32_t n, int32_t* scores, void* stream_) {
  DM_TRACE();
  if (!planes || !window || !samples || !scores) return DM_EINVAL;
  if (b <= 0 || C <= 0 || Hs <= 0 || Ws <= 0 || h <= 0 || w <= 0 || n <= 0 || !(map_res > 0.0f)) return DM_EINVAL;
  if (window_planes != 1 && window_planes != C) return DM_EINVAL;
  if ((long long)b * n >= (1ll << 31) || (long long)h * w >= (1ll << 31) || (long long)Hs * Ws >= (1ll << 31))
    return DM_EINVAL;
  if (reinterpret_cast<uintptr_t>(samples) % 4 != 0) return DM_EINVAL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long n_lists = (long long)b * window_planes;
  const long long hw = (long long)h * w;
  void* scratch = nullptr;                                // stream-ordered: the listed cells, then the counts
  DM_CUDA_OK(cudaMallocAsync(&scratch, (size_t)(n_lists * hw + n_lists) * sizeof(int), stream));
  int* cells = static_cast<int*>(scratch);
  int* counts = cells + n_lists * hw;
  const int pw = window_planes == 1 ? min(C, kPairs) : 1;           // planes per CTA
  const int plane_groups = window_planes == 1 ? (C + pw - 1) / pw : 1;
  const int G = kPairs / pw;                                        // candidates per CTA
  const int cand_groups = (n + G - 1) / G;
  const long long n_blocks = n_lists * plane_groups * cand_groups;
  const unsigned cap = 1u << 20;                                    // larger problems loop inside the kernels
  match_compact_kernel<<<(unsigned)min(n_lists, (long long)cap), kCompactThreads, 0, stream>>>(window, n_lists,
                                                                                                (int)hw, cells, counts);
  match_score_kernel<<<(unsigned)min(n_blocks, (long long)cap), kScoreThreads, 0, stream>>>(
      planes, C, Hs, Ws, map_res, flip_h, window_planes, h, w, samples, n, cells, counts, n_lists, plane_groups, pw,
      cand_groups, scores);
  const cudaError_t e = cudaGetLastError();
  DM_CUDA_OK(cudaFreeAsync(scratch, stream));
  DM_CUDA_OK(e);
  DM_LAUNCHED();
  return DM_OK;
}
