// distance_transform: per-plane exact Euclidean distance transform of bool masks (include/dungeon_maps_b200.h:
// dm_distance_transform_f32): for every cell, the distance to the nearest False cell of its plane and that cell, as
// scipy.ndimage.distance_transform_edt computes it.
//
// The separable exact transform (Meijster, Roerdink & Hesselink 2000; Felzenszwalb & Huttenlocher 2012).  The squared
// distance min over False cells (k, l) of (r - k)^2 + (c - l)^2 splits into a minimum along rows and one along
// columns, so the two passes may run in either order; here the row pass goes first because a warp reads a row with
// coalesced loads, and the column pass second because one thread per column then reads whole warp rows.  Passes, both
// on the caller's stream, no grid sync, no host sync, no atomics:
//   1. edt_rows_kernel  one warp per row: the column of the nearest False cell in the same row (ties: the left one),
//                       -1 when the row has none, into 2 B a cell of stream-ordered scratch.
//   2. edt_cols_kernel  one thread per column: the lower envelope of the parabolas (r - k)^2 + g(k)^2 over the rows k
//                       whose g (the pass-1 distance) is finite, then each cell's squared distance d2 and the cell that
//                       attains it.  Ties go to the smaller row, so the result is one fixed cell for every input.
// Everything is integer until d2 is final; dist = (float)sqrt((double)d2), the rounding scipy's float64 sqrt followed
// by .astype(float32) gives (sqrtf((float)d2) differs above 2^24).
#include "dm_common.cuh"

namespace dm {
namespace {

constexpr int kRowWarps = 4;                  // pass-1 CTA: 4 warps, one row each
constexpr int kColThreads = 128;              // pass-2 CTA: 128 columns
constexpr int kColPrefetch = 8;               // pass 2 loads the pass-1 columns of 8 rows at a time
constexpr int kNone = 1 << 30;                // "no False cell on this side" in pass 1

// Pass 1.  Per row, two sweeps of 32-cell chunks: right to left, the chunk's False bits (a ballot) and the first
// False cell right of the chunk go to shared memory; left to right, each lane takes the nearest False cell at or left
// of its cell (carried across chunks) and the nearest at or right of it.  Shared: 8 B per chunk per warp.
__global__ void __launch_bounds__(32 * kRowWarps) edt_rows_kernel(const uint8_t* __restrict__ mask, long long n_rows,
                                                                  int W, int16_t* __restrict__ near_col) {
  extern __shared__ unsigned smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kRowWarps + warp;
  if (row >= n_rows) return;                 // the whole warp: nothing below synchronises the block
  const int chunks = (W + 31) >> 5;
  unsigned* bits = smem + 2 * chunks * warp;
  int* right_of = reinterpret_cast<int*>(bits + chunks);
  const uint8_t* m = mask + row * W;
  int carry = kNone;                         // the first False column right of the current chunk
#pragma unroll 4
  for (int s = chunks - 1; s >= 0; --s) {
    const int c = 32 * s + lane;
    const unsigned w = __ballot_sync(0xffffffffu, c < W && !m[c]);
    if (lane == 0) {
      bits[s] = w;
      right_of[s] = carry;
    }
    if (w) carry = 32 * s + __ffs(w) - 1;
  }
  __syncwarp();
  int16_t* out = near_col + row * W;
  carry = -kNone;                            // the last False column left of the current chunk
  for (int s = 0; s < chunks; ++s) {
    const unsigned w = bits[s];
    const int c = 32 * s + lane;
    const unsigned le = w & (0xffffffffu >> (31 - lane)), ge = w >> lane;
    const int left = le ? 32 * s + 31 - __clz(le) : carry;
    const int right = ge ? c + __ffs(ge) - 1 : right_of[s];
    int col = c - left <= right - c ? left : right;
    if (col < 0 || col >= W) col = -1;       // neither side has one: the row is all True
    if (c < W) out[c] = (int16_t)col;
    if (w) carry = 32 * s + 31 - __clz(w);
  }
}

// Pass 2.  One column of one plane.  Sites are the rows k with a False cell in them (near_col >= 0); site k's parabola
// over rows r is f_k(r) = (r - k)^2 + g_k^2, g_k = c - near_col[k].  The envelope is a stack of (site, first row where
// it is the lowest) kept in the column's own cells of `env` (the dist buffer, as raw words): the stack never holds more
// entries than rows visited, and entry j starts at row >= j, so the fill that runs from the last row up overwrites
// only entries it has passed.  For sites v < u, u is strictly lower than v exactly on the rows r > sep(v, u) =
// floor(((u^2 + g_u^2) - (v^2 + g_v^2)) / (2 (u - v))) (numerators in int64); on rows <= sep the earlier site wins the
// tie.
__global__ void __launch_bounds__(kColThreads) edt_cols_kernel(const int16_t* __restrict__ near_col, long long n_cols,
                                                               int H, int W, unsigned* env, int2* __restrict__ nearest) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cols) return;
  const long long plane = t / W;
  const int c = (int)(t % W);
  const size_t base = (size_t)plane * H * W + c;
  const int16_t* g = near_col + base;        // row r at g[r * W]
  unsigned* st = env + base;                 // stack entry j at st[j * W]: site | start << 16
  int top = -1, v = 0, z = 0;                // the top entry, kept in registers
  long long fv = 0;                          // v^2 + g_v^2
  for (int u0 = 0; u0 < H; u0 += kColPrefetch) {
    int cols[kColPrefetch];                  // the next rows' pass-1 columns, loaded together
#pragma unroll
    for (int i = 0; i < kColPrefetch; ++i) cols[i] = u0 + i < H ? g[(size_t)(u0 + i) * W] : -1;
#pragma unroll
    for (int i = 0; i < kColPrefetch; ++i) {
      const int u = u0 + i, cu = cols[i];
      if (cu < 0) continue;
      const long long fu = (long long)u * u + (long long)(c - cu) * (c - cu);
      while (top >= 0 && fu - fv < (long long)z * 2 * (u - v)) {   // sep(v, u) < z: u is lower on all of v's rows
        if (--top >= 0) {
          const unsigned e = st[(size_t)top * W];
          v = (int)(e & 0xffffu);
          z = (int)(e >> 16);
          const int cv = g[(size_t)v * W];
          fv = (long long)v * v + (long long)(c - cv) * (c - cv);
        }
      }
      int start = 0;
      if (top >= 0) {
        const long long s = (fu - fv) / (2 * (u - v)) + 1;   // fu - fv >= 0 here
        if (s >= H) continue;                // u is never strictly lower inside the column
        start = (int)s;
      }
      ++top;
      v = u;
      z = start;
      fv = fu;
      st[(size_t)top * W] = (unsigned)u | (unsigned)start << 16;
    }
  }
  if (top < 0) {                             // no site: the plane has no False cell
    for (int r = 0; r < H; ++r) {
      st[(size_t)r * W] = 0x7f800000u;       // +inf
      if (nearest) nearest[base + (size_t)r * W] = make_int2(-1, -1);
    }
    return;
  }
  int cv = g[(size_t)v * W];
  for (int r = H - 1; r >= 0; --r) {
    if (z > r) {                             // entries start at increasing rows: one step down per row at most
      const unsigned e = st[(size_t)--top * W];
      v = (int)(e & 0xffffu);
      z = (int)(e >> 16);
      cv = g[(size_t)v * W];
    }
    const int dy = r - v, dx = c - cv;
    const int d2 = dy * dy + dx * dx;        // <= 2 * 32767^2 < 2^31
    st[(size_t)r * W] = __float_as_uint(__double2float_rn(sqrt((double)d2)));
    if (nearest) nearest[base + (size_t)r * W] = make_int2(cv, v);
  }
}

}  // namespace
}  // namespace dm

using namespace dm;

extern "C" int dm_distance_transform_f32(const uint8_t* mask, int32_t n_planes, int32_t H, int32_t W, float* dist,
                                         int32_t* nearest, void* stream_) {
  DM_TRACE();
  if (!mask || !dist || n_planes <= 0 || H <= 0 || W <= 0) return DM_EINVAL;
  if (H > 32768 || W > 32768) return DM_EINVAL;   // rows and columns fit 16 bits; d2 <= 2 * 32767^2 fits int32
  const long long n = (long long)n_planes * H * W;
  if (n > 0x7fffffffll) return DM_EINVAL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  void* scratch = nullptr;                   // stream-ordered: pass 1's nearest column per cell
  DM_CUDA_OK(cudaMallocAsync(&scratch, (size_t)n * sizeof(int16_t), stream));
  int16_t* near_col = static_cast<int16_t*>(scratch);
  const long long n_rows = (long long)n_planes * H, n_cols = (long long)n_planes * W;
  const size_t row_smem = (size_t)kRowWarps * 2 * ((W + 31) / 32) * sizeof(unsigned);   // <= 32 KB
  edt_rows_kernel<<<(unsigned)((n_rows + kRowWarps - 1) / kRowWarps), 32 * kRowWarps, row_smem, stream>>>(
      mask, n_rows, W, near_col);
  edt_cols_kernel<<<(unsigned)((n_cols + kColThreads - 1) / kColThreads), kColThreads, 0, stream>>>(
      near_col, n_cols, H, W, reinterpret_cast<unsigned*>(dist), reinterpret_cast<int2*>(nearest));
  const cudaError_t e = cudaGetLastError();
  DM_CUDA_OK(cudaFreeAsync(scratch, stream));
  DM_CUDA_OK(e);
  DM_LAUNCHED();
  return DM_OK;
}
