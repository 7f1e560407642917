// geodesic_distance: per-environment shortest-path distance fields over top-down maps (include/dungeon_maps_b200.h:
// dm_geodesic_distance_i32).  8-connected grid, orthogonal steps cost 5, diagonal steps 7, no corner cutting, an edge
// u -> v exists when v is traversable.  Integer costs: the result is exact and independent of evaluation order.
//
// One persistent cooperative launch.  The map is cut into 32 x 32 tiles; a CTA loads a tile with a one-cell halo into
// shared memory and relaxes it in place until it reaches its own fixed point for the halo it read (every stored value
// is the cost of a real path, so a racy read of a neighbour's value is an upper bound and is safe).  If a cell of the
// tile's outer ring changed, the tiles across that border are marked for the next round.  Rounds are separated by a
// grid-wide sync and the loop ends after a round that marked nothing: each tile then sits at the fixed point of halo
// values that have not changed since it last ran, so the Bellman equations hold everywhere and, with positive costs,
// have one solution.  The work follows the wavefront instead of sweeping the whole map every round.
//
// Round bound: after round k every cell whose shortest path crosses at most k tile borders is final (the tile it
// enters last was marked when the border cell before it became final).  A shortest path is simple, so it crosses at
// most H * W - 1 borders and H * W + 1 rounds always suffice.  Reaching that count means a bug: the kernel stops and
// raises the device's status word (dm_device_status reports DM_ETIMEOUT) instead of spinning.
#include <cooperative_groups.h>

#include "dm_project.cuh"

namespace dm {
namespace {
namespace cg = cooperative_groups;

constexpr int kTile = 32;
constexpr int kHalo = kTile + 2;
constexpr int kGeoThreads = 256;
constexpr int kCellsPerThread = kTile * kTile / kGeoThreads;  // rows ty, ty + 8, ty + 16, ty + 24 of column tx
constexpr int32_t kInf = 0x7fffffff;
constexpr int32_t kOrtho = 5;
constexpr int32_t kDiag = 7;

// border bits of a tile: which neighbour tiles read a changed cell as their halo
enum : int { kN = 1, kS = 2, kW = 4, kE = 8, kNW = 16, kNE = 32, kSW = 64, kSE = 128 };

struct GeoArgs {
  const uint8_t* trav;
  const uint8_t* src_mask;     // or nullptr
  const long long* src_cells;  // or nullptr: (b, n_cells, 2) [x, z]
  int n_cells, b, H, W, tiles_y, tiles_x;
  long long n_tiles;           // b * tiles_y * tiles_x
  long long max_rounds;
  int32_t* dist;
  uint8_t* flags;              // 2 * n_tiles: tiles to visit in even / odd rounds
  unsigned* any;               // 3 words: "a tile was marked" for the round after next, next, ... (rotating)
  uint32_t* status;            // mapped status word of the device, or nullptr
};

__device__ __forceinline__ int32_t relax(int32_t best, int32_t d, int32_t w) {
  return (d != kInf && d + w < best) ? d + w : best;
}

__device__ void relax_tile(const GeoArgs& a, long long t, int32_t (*sd)[kHalo], uint8_t (*st)[kHalo], int* s_mark,
                           uint8_t* next_flags, unsigned* any_next) {
  const int per_env = a.tiles_y * a.tiles_x;
  const int env = (int)(t / per_env);
  const int ty0 = (int)(t % per_env) / a.tiles_x * kTile, tx0 = (int)(t % per_env) % a.tiles_x * kTile;
  const size_t base = (size_t)env * a.H * a.W;
  for (int i = threadIdx.x; i < kHalo * kHalo; i += kGeoThreads) {
    const int r = i / kHalo, c = i % kHalo, gr = ty0 + r - 1, gc = tx0 + c - 1;
    const bool inside = gr >= 0 && gr < a.H && gc >= 0 && gc < a.W;
    const size_t g = base + (size_t)gr * a.W + gc;
    sd[r][c] = inside ? __ldcg(a.dist + g) : kInf;
    st[r][c] = inside ? a.trav[g] : 0;
  }
  if (threadIdx.x == 0) *s_mark = 0;
  __syncthreads();
  const int c = (threadIdx.x & 31) + 1, r0 = (threadIdx.x >> 5) + 1;
  int32_t orig[kCellsPerThread];
#pragma unroll
  for (int k = 0; k < kCellsPerThread; ++k) orig[k] = sd[r0 + 8 * k][c];
  bool changed;
  do {
    changed = false;
#pragma unroll
    for (int k = 0; k < kCellsPerThread; ++k) {
      const int r = r0 + 8 * k;
      if (!st[r][c]) continue;  // every edge into v needs T[v]: a blocked cell keeps 0 (source) or stays unreached
      const int32_t cur = sd[r][c];
      int32_t best = cur;
      best = relax(best, sd[r - 1][c], kOrtho);
      best = relax(best, sd[r + 1][c], kOrtho);
      best = relax(best, sd[r][c - 1], kOrtho);
      best = relax(best, sd[r][c + 1], kOrtho);
      const bool n = st[r - 1][c], s = st[r + 1][c], w = st[r][c - 1], e = st[r][c + 1];
      if (n && w) best = relax(best, sd[r - 1][c - 1], kDiag);
      if (n && e) best = relax(best, sd[r - 1][c + 1], kDiag);
      if (s && w) best = relax(best, sd[r + 1][c - 1], kDiag);
      if (s && e) best = relax(best, sd[r + 1][c + 1], kDiag);
      if (best < cur) {
        sd[r][c] = best;
        changed = true;
      }
    }
  } while (__syncthreads_or(changed));
  int sides = 0;
#pragma unroll
  for (int k = 0; k < kCellsPerThread; ++k) {
    const int r = r0 + 8 * k;
    if (sd[r][c] == orig[k]) continue;  // only cells inside the map can change (outside ones are not traversable)
    __stcg(a.dist + base + (size_t)(ty0 + r - 1) * a.W + (tx0 + c - 1), sd[r][c]);
    const bool top = r == 1, bottom = r == kTile, left = c == 1, right = c == kTile;
    sides |= (top ? kN : 0) | (bottom ? kS : 0) | (left ? kW : 0) | (right ? kE : 0) | (top && left ? kNW : 0) |
             (top && right ? kNE : 0) | (bottom && left ? kSW : 0) | (bottom && right ? kSE : 0);
  }
  if (sides) atomicOr(s_mark, sides);
  __syncthreads();
  const int mark = *s_mark;
  if (threadIdx.x < 8 && (mark >> threadIdx.x & 1)) {
    const int dy = (threadIdx.x == 0 || threadIdx.x == 4 || threadIdx.x == 5) ? -1
                   : (threadIdx.x == 1 || threadIdx.x == 6 || threadIdx.x == 7) ? 1 : 0;
    const int dx = (threadIdx.x == 2 || threadIdx.x == 4 || threadIdx.x == 6) ? -1
                   : (threadIdx.x == 3 || threadIdx.x == 5 || threadIdx.x == 7) ? 1 : 0;
    const int ty = ty0 / kTile + dy, tx = tx0 / kTile + dx;
    if (ty >= 0 && ty < a.tiles_y && tx >= 0 && tx < a.tiles_x) {
      __stcg(next_flags + (long long)env * per_env + ty * a.tiles_x + tx, (uint8_t)1);
      __stcg(any_next, 1u);
    }
  }
  __syncthreads();  // sd / st / s_mark are reused by the CTA's next tile
}

__global__ void __launch_bounds__(kGeoThreads) geodesic_kernel(const GeoArgs a) {
  __shared__ int32_t sd[kHalo][kHalo];
  __shared__ uint8_t st[kHalo][kHalo];
  __shared__ int s_mark;
  cg::grid_group grid = cg::this_grid();
  const long long gtid = (long long)blockIdx.x * kGeoThreads + threadIdx.x;
  const long long gstride = (long long)gridDim.x * kGeoThreads;
  const long long total = (long long)a.b * a.H * a.W;
  for (long long i = gtid; i < total; i += gstride) a.dist[i] = (a.src_mask && a.src_mask[i]) ? 0 : kInf;
  for (long long t = gtid; t < a.n_tiles; t += gstride) {
    a.flags[t] = 1;  // round 0 visits every tile
    a.flags[a.n_tiles + t] = 0;
  }
  if (gtid < 3) a.any[gtid] = 0u;
  if (a.src_cells) {
    grid.sync();
    for (long long k = gtid; k < (long long)a.b * a.n_cells; k += gstride) {
      const long long x = a.src_cells[2 * k], z = a.src_cells[2 * k + 1];
      if (x >= 0 && x < a.W && z >= 0 && z < a.H) a.dist[(size_t)(k / a.n_cells) * a.H * a.W + z * a.W + x] = 0;
    }
  }
  grid.sync();
  for (long long round = 0;; ++round) {
    uint8_t* cur = a.flags + (round & 1) * a.n_tiles;
    uint8_t* next = a.flags + ((round + 1) & 1) * a.n_tiles;
    unsigned* any_next = a.any + (round + 1) % 3;
    // the word of round + 2 was last read right after the previous grid sync, by every thread
    if (gtid == 0) a.any[(round + 2) % 3] = 0u;
    for (long long t = blockIdx.x; t < a.n_tiles; t += gridDim.x) {
      if (!__ldcg(cur + t)) continue;  // uniform in the CTA: nobody writes this round's flags during the round
      __syncthreads();
      if (threadIdx.x == 0) cur[t] = 0;
      relax_tile(a, t, sd, st, &s_mark, next, any_next);
    }
    grid.sync();
    if (__ldcg(any_next) == 0u) break;
    if (round + 1 >= a.max_rounds) {
      if (gtid == 0 && a.status) asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(a.status), "r"(1u) : "memory");
      break;
    }
  }
  for (long long i = gtid; i < total; i += gstride)
    if (__ldcg(a.dist + i) == kInf) a.dist[i] = -1;
}

// geodesic_path (dm_geodesic_path_i32): the walk down a field D from a start s.  p_0 = s when s is inside the map and
// D[s] >= 0 (else the path is empty); while D[p_k] > 0 and k + 1 < max_cells, p_k+1 is the first neighbour
// q = p_k + (dx, dz), in the order (+1, 0), (0, +1), (-1, 0), (0, -1), (+1, +1), (-1, +1), (-1, -1), (+1, -1), inside
// the map with D[q] >= 0, D[q] == D[p_k] - cost and an edge q -> p_k under geodesic_kernel's rule (T[p_k], and for a
// diagonal step T of both side cells).  D strictly decreases along the walk, so it ends for any int32 field.
//
// One warp per (environment, start).  Lanes 0..7 own the 8 neighbours in the definition's order and load D and T of
// theirs together through the read-only path (consecutive steps share most of their 3 x 3 neighbourhood, so they
// mostly hit L1); the first qualifying neighbour is the lowest set bit of a ballot.  Lane k % 32 keeps cell k, and
// each group of 32 cells is stored as one coalesced 256-byte row; the warp then fills the rest of the path with -1.
constexpr int kPathThreads = 256;
constexpr int kPathWarps = kPathThreads / 32;

struct PathArgs {
  const uint8_t* trav;       // (b, H, W)
  const int32_t* dist;       // (b, H, W)
  const long long* starts;   // (b, n, 2) [x, z]
  int H, W, n, max_cells;
  long long paths;           // b * n
  int2* cells;               // (b, n, max_cells) [x, z]
  int32_t* lengths;          // (b, n)
};

__global__ void __launch_bounds__(kPathThreads) geodesic_path_kernel(const PathArgs a) {
  const int lane = threadIdx.x & 31;
  const long long path = (long long)blockIdx.x * kPathWarps + (threadIdx.x >> 5);
  if (path >= a.paths) return;                             // uniform in the warp
  // lane j < 8 owns the j-th neighbour of the order above; lanes >= 8 only store
  const int dx = (lane == 0 || lane == 4 || lane == 7) ? 1 : (lane == 2 || lane == 5 || lane == 6) ? -1 : 0;
  const int dz = (lane == 1 || lane == 4 || lane == 5) ? 1 : (lane == 3 || lane == 6 || lane == 7) ? -1 : 0;
  const bool diag = dx != 0 && dz != 0;
  const int32_t cost = diag ? kDiag : kOrtho;
  // a diagonal step needs T of its side cells (q.x, p.z) = p + (dx, 0) and (p.x, q.z) = p + (0, dz): lanes 0 / 2, 1 / 3
  const unsigned sides = diag ? (1u << (dx > 0 ? 0 : 2)) | (1u << (dz > 0 ? 1 : 3)) : 0u;
  const size_t plane = (size_t)(path / a.n) * a.H * a.W;
  const int32_t* D = a.dist + plane;
  const uint8_t* T = a.trav + plane;
  int2* out = a.cells + path * a.max_cells;
  const long long sx = a.starts[2 * path], sz = a.starts[2 * path + 1];
  int len = 0;
  const bool inside = sx >= 0 && sx < a.W && sz >= 0 && sz < a.H;
  int32_t d = inside ? __ldg(D + sz * a.W + sx) : -1;
  if (d >= 0) {
    int x = (int)sx, z = (int)sz;
    bool t = __ldg(T + sz * a.W + sx) != 0;
    int2 mine = make_int2(-1, -1);                         // cell k of the walk, k % 32 == lane
    int k = 0;
    for (;;) {
      if (lane == (k & 31)) mine = make_int2(x, z);
      if ((k & 31) == 31) out[k - 31 + lane] = mine;
      if (d == 0 || k + 1 >= a.max_cells || !t) break;     // a source, the capacity, or no edge into p_k
      const int qx = x + dx, qz = z + dz;
      int32_t dq = -1;
      bool tq = false;
      if (lane < 8 && qx >= 0 && qx < a.W && qz >= 0 && qz < a.H) {
        const size_t g = (size_t)qz * a.W + qx;
        dq = __ldg(D + g);
        tq = __ldg(T + g) != 0;
      }
      const unsigned tb = __ballot_sync(0xffffffffu, tq);
      const bool ok = dq >= 0 && dq == d - cost && (tb & sides) == sides;   // d > 0: d - cost cannot overflow
      const unsigned win = __ballot_sync(0xffffffffu, ok);
      if (!win) break;
      const int w = __ffs(win) - 1;
      x = __shfl_sync(0xffffffffu, qx, w);
      z = __shfl_sync(0xffffffffu, qz, w);
      d = __shfl_sync(0xffffffffu, dq, w);
      t = (tb >> w) & 1u;
      ++k;
    }
    len = k + 1;
    if ((k & 31) != 31 && lane <= (k & 31)) out[(k & ~31) + lane] = mine;
  }
  for (long long i = len + lane; i < a.max_cells; i += 32) out[i] = make_int2(-1, -1);
  if (lane == 0) a.lengths[path] = len;
}
}  // namespace
}  // namespace dm

using namespace dm;

extern "C" int dm_geodesic_distance_i32(const uint8_t* traversable, const uint8_t* source_mask,
                                        const int64_t* source_cells, int32_t n_cells, int32_t b, int32_t H, int32_t W,
                                        int32_t* dist, void* stream_) {
  DM_TRACE();
  if (!traversable || !dist || b <= 0 || H <= 0 || W <= 0) return DM_EINVAL;
  if (!source_mask == !source_cells) return DM_EINVAL;                 // exactly one source form
  if (source_cells ? n_cells <= 0 : n_cells != 0) return DM_EINVAL;
  if (7ll * H * W > 0x7fffffffll) return DM_EINVAL;                    // the largest distance must fit in int32
  const int tiles_y = (H + kTile - 1) / kTile, tiles_x = (W + kTile - 1) / kTile;
  const long long n_tiles = (long long)b * tiles_y * tiles_x;
  if (n_tiles >= (1ll << 31)) return DM_EINVAL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int device = 0, per_sm = 0;
  DM_CUDA_OK(cudaGetDevice(&device));
  DM_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, geodesic_kernel, kGeoThreads, 0));
  if (per_sm < 1) return DM_EINVAL;
  long long grid = (long long)sm_count() * per_sm;
  if (grid > n_tiles) grid = n_tiles;
  GeoArgs a;
  a.trav = traversable;
  a.src_mask = source_mask;
  a.src_cells = reinterpret_cast<const long long*>(source_cells);
  a.n_cells = source_cells ? n_cells : 0;
  a.b = b;
  a.H = H;
  a.W = W;
  a.tiles_y = tiles_y;
  a.tiles_x = tiles_x;
  a.n_tiles = n_tiles;
  a.max_rounds = (long long)H * W + 2;
  a.dist = dist;
  a.status = proj_guard(device).status;
  void* scratch = nullptr;  // stream-ordered: the tile flags and the three round words
  const size_t flag_bytes = (size_t)(2 * n_tiles + 15) / 16 * 16;
  DM_CUDA_OK(cudaMallocAsync(&scratch, flag_bytes + 3 * sizeof(unsigned), stream));
  a.flags = static_cast<uint8_t*>(scratch);
  a.any = reinterpret_cast<unsigned*>(a.flags + flag_bytes);
  void* params[] = {&a};
  const cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(geodesic_kernel), dim3((unsigned)grid),
                                                    dim3(kGeoThreads), params, 0, stream);
  DM_CUDA_OK(cudaFreeAsync(scratch, stream));
  DM_CUDA_OK(e);
  DM_LAUNCHED();
  return DM_OK;
}

extern "C" int dm_geodesic_path_i32(const uint8_t* traversable, const int32_t* dist, int32_t b, int32_t H, int32_t W,
                                    const int64_t* starts, int32_t n, int32_t max_cells, int32_t* cells,
                                    int32_t* lengths, void* stream_) {
  DM_TRACE();
  if (!traversable || !dist || !starts || !cells || !lengths) return DM_EINVAL;
  if (b <= 0 || H <= 0 || W <= 0 || n <= 0) return DM_EINVAL;
  const long long HW = (long long)H * W, paths = (long long)b * n;
  if (HW >= (1ll << 31) || paths >= (1ll << 31)) return DM_EINVAL;
  if (max_cells < 1 || max_cells > HW) return DM_EINVAL;
  PathArgs a;
  a.trav = traversable;
  a.dist = dist;
  a.starts = reinterpret_cast<const long long*>(starts);
  a.H = H;
  a.W = W;
  a.n = n;
  a.max_cells = max_cells;
  a.paths = paths;
  a.cells = reinterpret_cast<int2*>(cells);
  a.lengths = lengths;
  const long long blocks = (paths + kPathWarps - 1) / kPathWarps;
  geodesic_path_kernel<<<(unsigned)blocks, kPathThreads, 0, static_cast<cudaStream_t>(stream_)>>>(a);
  DM_LAUNCHED();
  return DM_OK;
}
