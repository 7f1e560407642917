// connected_components: per-plane connected-component labels of bool masks (include/dungeon_maps_b200.h:
// dm_connected_components_i32), numbered 1..K in raster order of each component's first cell, as scipy.ndimage.label
// numbers them.
//
// Block-based union-find (Playne & Hawick 2018; Allegretti et al. 2019).  While the components are being joined,
// `labels` holds a parent per cell as a plane-linear index (-1 on background).  Every union links the larger of two
// roots under the smaller with atomicMin, so parent[i] <= i always holds: a find loop walks a strictly decreasing
// chain and ends, and the root a component ends with is its smallest index, its first cell in raster order, whatever
// order the atomics ran in.  Passes, all on the caller's stream, no grid sync and no host sync:
//   1. cc_tile_kernel     one CTA per 32 x 32 tile: union-find of the tile in shared memory, parents written out
//   2. cc_border_kernel   one thread per tile-border cell: unions with its neighbours in other tiles, in global memory
//   3. cc_flatten_kernel  every cell points at its root; flags the roots; counts the cells per root (sizes only)
//   4. cub exclusive sum  of the root flags: the rank of each root among all roots before it
//   5. cc_number_kernel   label = rank(root) - rank(plane start) + 1, the plane's component count, the sizes gathered
#include <cub/device/device_scan.cuh>

#include "dm_common.cuh"

namespace dm {
namespace {

constexpr int kCcTile = 32;
constexpr int kCcRows = 8;                    // a 32 x 8 CTA; each thread takes rows ty, ty + 8, ty + 16, ty + 24
constexpr int kCcThreads = kCcTile * kCcRows;
constexpr int kBorderCells = 3 * kCcTile;     // per tile: its top row, left column and right column

__device__ __forceinline__ int find_shared(const volatile int* p, int a) {
  for (int q = p[a]; q != a; q = p[a]) a = q;
  return a;
}

// p: parents of one plane (or tile).  Joins the sets of a and b; on return they share a root.  An atomicMin that
// finds its target no longer a root still lowers it within the same component, and the loop retries from the value it
// found, which is strictly smaller: the loop ends.
template <bool kShared>
__device__ void unite(int* p, int a, int b) {
  for (;;) {
    if (kShared) {
      a = find_shared(p, a);
      b = find_shared(p, b);
    } else {
      for (int q = __ldcg(p + a); q != a; q = __ldcg(p + a)) a = q;
      for (int q = __ldcg(p + b); q != b; q = __ldcg(p + b)) b = q;
    }
    if (a == b) return;
    if (a < b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(p + a, b);  // a > b: the larger root goes under the smaller
    if (old == a) return;
    a = old;
  }
}

__global__ void __launch_bounds__(kCcThreads) cc_tile_kernel(const uint8_t* __restrict__ mask, int H, int W,
                                                             int tiles_x, int tiles_per_plane, int conn,
                                                             int* __restrict__ labels) {
  __shared__ int sp[kCcTile * kCcTile];      // tile-local parents, row-major in the tile (-1: background)
  const int plane = blockIdx.x / tiles_per_plane, t = blockIdx.x % tiles_per_plane;
  const int ty0 = t / tiles_x * kCcTile, tx0 = t % tiles_x * kCcTile;
  const int th = min(kCcTile, H - ty0), tw = min(kCcTile, W - tx0);
  const size_t base = (size_t)plane * H * W;
  const int c = threadIdx.x;
#pragma unroll
  for (int k = 0; k < kCcTile / kCcRows; ++k) {
    const int r = threadIdx.y + kCcRows * k;
    const bool fg = r < th && c < tw && mask[base + (size_t)(ty0 + r) * W + tx0 + c];
    sp[r * kCcTile + c] = fg ? r * kCcTile + c : -1;
  }
  __syncthreads();
  // each edge once, from its later cell: W and N, and for 8-connectivity NW and NE
#pragma unroll
  for (int k = 0; k < kCcTile / kCcRows; ++k) {
    const int r = threadIdx.y + kCcRows * k, i = r * kCcTile + c;
    if (sp[i] < 0) continue;
    if (c > 0 && sp[i - 1] >= 0) unite<true>(sp, i, i - 1);
    if (r > 0) {
      if (sp[i - kCcTile] >= 0) unite<true>(sp, i, i - kCcTile);
      if (conn == 8 && c > 0 && sp[i - kCcTile - 1] >= 0) unite<true>(sp, i, i - kCcTile - 1);
      if (conn == 8 && c + 1 < kCcTile && sp[i - kCcTile + 1] >= 0) unite<true>(sp, i, i - kCcTile + 1);
    }
  }
  __syncthreads();
  // tile row-major order agrees with plane raster order, so the tile's smallest root is also the plane's smallest
#pragma unroll
  for (int k = 0; k < kCcTile / kCcRows; ++k) {
    const int r = threadIdx.y + kCcRows * k, i = r * kCcTile + c;
    if (r >= th || c >= tw) continue;
    int v = -1;
    if (sp[i] >= 0) {
      const int root = find_shared(sp, i);
      v = (ty0 + root / kCcTile) * W + tx0 + root % kCcTile;
    }
    labels[base + (size_t)(ty0 + r) * W + tx0 + c] = v;
  }
}

__global__ void __launch_bounds__(256) cc_border_kernel(int H, int W, int tiles_x, int tiles_per_plane,
                                                        long long n_tiles, int conn, int* labels) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_tiles * kBorderCells) return;
  const int tile = (int)(g / kBorderCells), k = (int)(g % kBorderCells);
  const int side = k / kCcTile, j = k % kCcTile;
  if (side == 2 && conn == 4) return;        // the right column's only edge out of the tile is NE
  const int plane = tile / tiles_per_plane, t = tile % tiles_per_plane;
  const int r = side == 0 ? 0 : j, c = side == 0 ? j : side == 1 ? 0 : kCcTile - 1;
  const int gr = t / tiles_x * kCcTile + r, gc = t % tiles_x * kCcTile + c;
  if (gr >= H || gc >= W) return;
  int* p = labels + (size_t)plane * H * W;
  const int i = gr * W + gc;
  if (p[i] < 0) return;
  // the neighbours before this cell (W, N, NW, NE) that lie in another tile
  if (c == 0 && gc > 0 && p[i - 1] >= 0) unite<false>(p, i, i - 1);
  if (gr == 0) return;
  if (r == 0 && p[i - W] >= 0) unite<false>(p, i, i - W);
  if (conn == 4) return;
  if ((r == 0 || c == 0) && gc > 0 && p[i - W - 1] >= 0) unite<false>(p, i, i - W - 1);
  if ((r == 0 || c == kCcTile - 1) && gc + 1 < W && p[i - W + 1] >= 0) unite<false>(p, i, i - W + 1);
}

__global__ void __launch_bounds__(256) cc_flatten_kernel(long long n, int plane_cells, int* labels, int* is_root,
                                                         int* sizes) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  int* p = labels + g / plane_cells * plane_cells;
  const int i = (int)(g % plane_cells);
  const int parent = p[i];
  int a = parent, flag = 0;
  if (a >= 0) {
    for (int q = __ldcg(p + a); q != a; q = __ldcg(p + a)) a = q;
    if (a != parent) p[i] = a;               // another ancestor: a racing reader follows either value to the same root
    flag = a == i;
    if (sizes) atomicAdd(sizes + (g - i) + a, 1);
  }
  is_root[g] = flag;
}

__global__ void __launch_bounds__(256) cc_number_kernel(long long n, int plane_cells, int* labels, const int* rank,
                                                        int* counts, int* sizes) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  const int i = (int)(g % plane_cells);
  const long long start = g - i;
  const int a = labels[g];                   // the root, or -1; no other thread reads this cell any more
  const int first = rank[start];
  labels[g] = a >= 0 ? rank[start + a] - first + 1 : 0;
  if (sizes && a >= 0 && a != i) sizes[g] = sizes[start + a];   // the root's entry holds its count and stays
  if (i == plane_cells - 1) counts[g / plane_cells] = rank[g] + (a == i) - first;
}

}  // namespace
}  // namespace dm

using namespace dm;

extern "C" int dm_connected_components_i32(const uint8_t* mask, int32_t n_planes, int32_t H, int32_t W,
                                           int32_t connectivity, int32_t* labels, int32_t* counts, int32_t* sizes,
                                           void* stream_) {
  DM_TRACE();
  if (!mask || !labels || !counts || n_planes <= 0 || H <= 0 || W <= 0) return DM_EINVAL;
  if (connectivity != 4 && connectivity != 8) return DM_EINVAL;
  const long long n = (long long)n_planes * H * W;
  if (n > 0x7fffffffll) return DM_EINVAL;    // plane-linear parents, the ranks and the scan's length are int32
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int tiles_y = (H + kCcTile - 1) / kCcTile, tiles_x = (W + kCcTile - 1) / kCcTile;
  const int tiles_per_plane = tiles_y * tiles_x;   // <= H * W
  const long long n_tiles = (long long)n_planes * tiles_per_plane;   // <= n
  size_t scan_bytes = 0;
  DM_CUDA_OK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, static_cast<int*>(nullptr), static_cast<int*>(nullptr),
                                           (int)n, stream));
  const size_t rank_bytes = ((size_t)n * sizeof(int) + 255) / 256 * 256;
  void* scratch = nullptr;                   // stream-ordered: the root flags, scanned in place into ranks, and cub's
  DM_CUDA_OK(cudaMallocAsync(&scratch, rank_bytes + scan_bytes, stream));
  int* rank = static_cast<int*>(scratch);
  void* cub_temp = static_cast<uint8_t*>(scratch) + rank_bytes;
  const unsigned cell_blocks = (unsigned)((n + 255) / 256);
  cudaError_t e = cudaSuccess;
  if (sizes) e = cudaMemsetAsync(sizes, 0, (size_t)n * sizeof(int32_t), stream);
  if (e == cudaSuccess) {
    cc_tile_kernel<<<(unsigned)n_tiles, dim3(kCcTile, kCcRows), 0, stream>>>(mask, H, W, tiles_x, tiles_per_plane,
                                                                              connectivity, labels);
    cc_border_kernel<<<(unsigned)((n_tiles * kBorderCells + 255) / 256), 256, 0, stream>>>(
        H, W, tiles_x, tiles_per_plane, n_tiles, connectivity, labels);
    cc_flatten_kernel<<<cell_blocks, 256, 0, stream>>>(n, H * W, labels, rank, sizes);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(cub_temp, scan_bytes, rank, rank, (int)n, stream);
  if (e == cudaSuccess) {
    cc_number_kernel<<<cell_blocks, 256, 0, stream>>>(n, H * W, labels, rank, counts, sizes);
    e = cudaGetLastError();
  }
  DM_CUDA_OK(cudaFreeAsync(scratch, stream));
  DM_CUDA_OK(e);
  DM_LAUNCHED();
  return DM_OK;
}
